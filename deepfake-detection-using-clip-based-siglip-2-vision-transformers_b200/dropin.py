"""Drop-in Python surface of the detection hot path (SURVEY.md §8b): the names, arguments and return shapes the
reference's entry points use, backed by the dfd engine instead of open_clip / timm / HF modules.

    open_clip.create_model_and_transforms(name, pretrained, device) -> (model, None, preprocess)
        inference_ai_human_images.py:124-128, train_fusion_head_only.py:81-83, coral.py:87-89
    BinaryClassifier(model_size, device)  .backbone .preprocess .resolution .classifier  forward(x) -> [B]
        inference_ai_human_images.py:111-152 (head H-A) ; train_fusion_head_only.py:78-109 (SE + head H-B)
    run_inference / few_shot_prototype
        inference_ai_human_images.py:250-318, 477-541
    transformers.SiglipVisionModel(...)(pixel_values=...) -> .pooler_output / .last_hidden_state
        Siglip2sidafrozen.py:753,787-788

`install_import_shims()` registers `open_clip` and `pywt` stand-ins in sys.modules so the reference scripts can be
imported unmodified on a box without those packages.
"""
from __future__ import annotations

import os
import sys
import types
import warnings
from typing import Dict, Iterable, Optional

import numpy as np
import torch
import torch.nn as nn
from torch.nn.modules.module import _IncompatibleKeys

from . import ops
from .engine import ARCHS, SiglipEngine, VisionArch, arch_from_state_dict, canonicalize_state_dict
from .pipeline import head_params_from_state
from .weights import random_classifier_head, random_vision_state_dict


def _as_device(device) -> torch.device:
    d = torch.device(device)
    if d.type != "cuda":
        raise RuntimeError("the dfd backbone runs on CUDA only (sm_100a); there is no CPU fallback")
    return torch.device("cuda", d.index if d.index is not None else torch.cuda.current_device())


def make_preprocess(resolution: int, interpolation: str = "bicubic"):
    """PIL -> float32 [3,S,S] in [-1,1]: Resize((S,S)) + ToTensor + Normalize(.5,.5) — what open_clip's SigLIP
    transform and inference_ai_human_images.py:200-204 produce.  (Host side, as in the reference.)"""
    from torchvision import transforms
    from torchvision.transforms import InterpolationMode

    mode = {"bicubic": InterpolationMode.BICUBIC, "bilinear": InterpolationMode.BILINEAR}[interpolation]
    return transforms.Compose([
        transforms.Lambda(lambda im: im.convert("RGB")),
        transforms.Resize((resolution, resolution), interpolation=mode),
        transforms.ToTensor(),
        transforms.Normalize([0.5] * 3, [0.5] * 3),
    ])


# ---------------------------------------------------------------------------------------------------------------------
# open_clip-shaped vision tower: a real nn.Module whose registered parameters carry the timm names of open_clip's SigLIP
# models (visual.trunk.blocks.i.attn.qkv.weight, visual.trunk.attn_pool.*, visual.trunk.pos_embed, ...), so that the
# reference's OWN classes - BinaryClassifier(nn.Module) of inference_ai_human_images.py:111-152 and
# train_fusion_head_only.py:78-109 - register it as a submodule and their load_state_dict(strict=True) /
# _filter_state_for_model route the checkpoint's `backbone.*` tensors into it.  The parameters are the source of truth;
# the dfd engine keeps a packed bf16 copy that is refreshed whenever they change (load_state_dict, in-place updates).
# ---------------------------------------------------------------------------------------------------------------------
class _Holder(nn.Module):
    """Parameter container with the reference model's attribute names; never called (the dfd engine runs the math)."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("dfd: this module only holds parameters; call the tower's encode_image()")


def _linear(out_f: int, in_f: int) -> nn.Module:
    m = _Holder()
    m.weight = nn.Parameter(torch.empty(out_f, in_f), requires_grad=False)
    m.bias = nn.Parameter(torch.empty(out_f), requires_grad=False)
    return m


def _norm(dim: int) -> nn.Module:
    m = _Holder()
    m.weight = nn.Parameter(torch.empty(dim), requires_grad=False)
    m.bias = nn.Parameter(torch.empty(dim), requires_grad=False)
    return m


def _timm_trunk(a: VisionArch) -> nn.Module:
    """Skeleton of timm's VisionTransformer(global_pool='map') as open_clip builds it for SigLIP (SURVEY.md App. B)."""
    D, I, P, N = a.hidden_size, a.intermediate_size, a.patch_size, a.tokens
    trunk = _Holder()
    trunk.patch_embed = _Holder()
    trunk.patch_embed.proj = _Holder()
    trunk.patch_embed.proj.weight = nn.Parameter(torch.empty(D, 3, P, P), requires_grad=False)
    trunk.patch_embed.proj.bias = nn.Parameter(torch.empty(D), requires_grad=False)
    trunk.pos_embed = nn.Parameter(torch.empty(1, N, D), requires_grad=False)
    blocks = []
    for _ in range(a.num_hidden_layers):
        b = _Holder()
        b.norm1, b.norm2 = _norm(D), _norm(D)
        b.attn = _Holder()
        b.attn.qkv, b.attn.proj = _linear(3 * D, D), _linear(D, D)
        b.mlp = _Holder()
        b.mlp.fc1, b.mlp.fc2 = _linear(I, D), _linear(D, I)
        blocks.append(b)
    trunk.blocks = nn.ModuleList(blocks)
    trunk.norm = _norm(D)
    ap = _Holder()
    ap.latent = nn.Parameter(torch.empty(1, 1, D), requires_grad=False)
    ap.q, ap.kv, ap.proj, ap.norm = _linear(D, D), _linear(2 * D, D), _linear(D, D), _norm(D)
    ap.mlp = _Holder()
    ap.mlp.fc1, ap.mlp.fc2 = _linear(I, D), _linear(D, I)
    trunk.attn_pool = ap
    return trunk


def timm_state_from_canonical(canon: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Engine-canonical (HF-style) vision tensors -> open_clip/timm names under `visual.trunk.` (inverse of
    engine.canonicalize_state_dict for that layout)."""
    out: Dict[str, torch.Tensor] = {}
    T = "visual.trunk."
    out[T + "patch_embed.proj.weight"] = canon["embeddings.patch_embedding.weight"]
    out[T + "patch_embed.proj.bias"] = canon["embeddings.patch_embedding.bias"]
    pe = canon["embeddings.position_embedding.weight"]
    out[T + "pos_embed"] = pe.reshape(1, pe.shape[-2], pe.shape[-1])
    L = 1 + max(int(k.split(".")[2]) for k in canon if k.startswith("encoder.layers."))
    for i in range(L):
        s, d = f"encoder.layers.{i}.", f"{T}blocks.{i}."
        for n in ("weight", "bias"):
            out[d + "norm1." + n] = canon[s + "layer_norm1." + n]
            out[d + "norm2." + n] = canon[s + "layer_norm2." + n]
            if s + "self_attn.qkv." + n in canon:
                out[d + "attn.qkv." + n] = canon[s + "self_attn.qkv." + n]
            else:
                out[d + "attn.qkv." + n] = torch.cat([canon[s + f"self_attn.{x}_proj." + n] for x in "qkv"], 0)
            out[d + "attn.proj." + n] = canon[s + "self_attn.out_proj." + n]
            out[d + "mlp.fc1." + n] = canon[s + "mlp.fc1." + n]
            out[d + "mlp.fc2." + n] = canon[s + "mlp.fc2." + n]
    for n in ("weight", "bias"):
        out[T + "norm." + n] = canon["post_layernorm." + n]
        out[T + "attn_pool.proj." + n] = canon["head.attention.out_proj." + n]
        out[T + "attn_pool.norm." + n] = canon["head.layernorm." + n]
        out[T + "attn_pool.mlp.fc1." + n] = canon["head.mlp.fc1." + n]
        out[T + "attn_pool.mlp.fc2." + n] = canon["head.mlp.fc2." + n]
    D = pe.shape[-1]
    out[T + "attn_pool.latent"] = canon["head.probe"].reshape(1, 1, D)
    w, b = canon["head.attention.in_proj_weight"], canon["head.attention.in_proj_bias"]
    out[T + "attn_pool.q.weight"], out[T + "attn_pool.kv.weight"] = w[:D], w[D:]
    out[T + "attn_pool.q.bias"], out[T + "attn_pool.kv.bias"] = b[:D], b[D:]
    return out


class _TextSink(nn.Module):
    """Stands where open_clip keeps the text tower: swallows `text.*` checkpoint keys (the reference drops them,
    train_fusion_head_only.py:115) so that a strict load of a full open_clip checkpoint still succeeds."""

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        return


class VisionTower(nn.Module):
    """What `open_clip.create_model_and_transforms` returns, reduced to what the reference touches: an nn.Module with
    `encode_image`, `embed_dim`, `visual.trunk.*` parameters (timm names), `eval/to/parameters/state_dict/
    load_state_dict`.  The forward runs on the dfd engine (hand-written sm_100a kernels); there is no torch fallback."""

    def __init__(self, arch: VisionArch, device, max_batch: int = 64, state_dict: Optional[dict] = None, seed: int = 0,
                 fuse_ln: bool = True):
        super().__init__()
        self.arch = arch
        d = torch.device(device)
        # Without a CUDA device only the parameter skeleton exists (state-dict round trips work, e.g. to inspect or
        # convert checkpoints); every forward raises - there is no CPU fallback.
        self._device = _as_device(d) if d.type == "cuda" else d
        self.embed_dim = arch.hidden_size
        self.resize_mode = ops.RESIZE_NONE
        self.visual = _Holder()
        self.visual.trunk = _timm_trunk(arch)
        self.visual.image_size = (arch.image_size, arch.image_size)
        self.text = _TextSink()
        self.to_empty(device=self._device)
        self.engine = (SiglipEngine(arch, self._device.index, max_batch, fuse_ln=fuse_ln)
                       if self._device.type == "cuda" else None)
        self._synced = None                 # parameter-version fingerprint the engine's packed copy corresponds to
        self.weights_source = "random"      # "random" until real tensors arrive through load_state_dict
        self._warned_random = False
        src = state_dict if state_dict is not None else random_vision_state_dict(arch, seed, device=self._device)
        canon = canonicalize_state_dict(src)
        own = timm_state_from_canonical(canon)
        with torch.no_grad():
            params = dict(self.named_parameters())
            for k, v in own.items():
                params[k].copy_(v.to(self._device, torch.float32).reshape(params[k].shape))
        if state_dict is not None:
            self.weights_source = "state_dict"
        self.register_load_state_dict_post_hook(VisionTower._after_load)

    # ---- state dict plumbing -------------------------------------------------------------------------------------
    _IGNORED_TOP = ("logit_scale", "logit_bias")

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        # the tower itself owns no tensors; open_clip's scalar `logit_scale` / `logit_bias` are accepted and dropped, and
        # HF-layout keys (`vision_model.*`) are translated so either checkpoint flavour loads through the same path
        hf = {k[len(prefix):]: v for k, v in state_dict.items()
              if k.startswith(prefix + "vision_model.") or k.startswith(prefix + "visual.vision_model.")}
        if hf:
            own = timm_state_from_canonical(canonicalize_state_dict(hf))
            for k in list(state_dict.keys()):
                if k.startswith(prefix + "vision_model.") or k.startswith(prefix + "visual.vision_model."):
                    del state_dict[k]
            for k, v in own.items():
                state_dict[prefix + k] = v
        if strict:
            for key in state_dict.keys():
                if key.startswith(prefix):
                    head = key[len(prefix):].split(".", 1)[0]
                    if head not in ("visual", "text") and head not in self._IGNORED_TOP:
                        unexpected_keys.append(key)

    @staticmethod
    def _after_load(module, incompatible_keys):
        missing = [k for k in incompatible_keys.missing_keys if "visual.trunk." in k]
        total = sum(1 for _ in module.visual.trunk.parameters())
        if len(missing) < total:   # at least part of the backbone arrived
            module.weights_source = "checkpoint" if not missing else "checkpoint (partial)"
            if missing:
                warnings.warn(f"dfd: {len(missing)} of {total} backbone tensors were not in the checkpoint and keep their "
                              f"previous values (first: {missing[0]})", stacklevel=2)
        module._synced = None

    def _fingerprint(self):
        ps = list(self.visual.trunk.parameters())
        try:
            vers = tuple(p._version for p in ps)
        except RuntimeError:   # inference tensors carry no version counter: storage identity only
            vers = ()
        return vers + tuple(p.data_ptr() for p in ps)

    def sync_engine(self, force: bool = False) -> None:
        """Repack the registered parameters into the engine if they changed since the last forward."""
        if self.engine is None:
            raise RuntimeError("dfd: the vision tower was created without a CUDA device; the backbone has no CPU fallback")
        fp = self._fingerprint()
        if force or fp != self._synced:
            sd = {"visual.trunk." + k: v.detach() for k, v in self.visual.trunk.named_parameters()}
            self.engine.load_state_dict(sd)
            self._synced = fp

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        p = next(self.visual.trunk.parameters(), None)
        if p is not None and p.device != self._device and self.engine is not None:
            raise RuntimeError(f"dfd: the vision tower lives on {self._device}; moving it to {p.device} is not supported "
                               "(the engine's workspace and packed weights stay on the device it was created on)")
        self._synced = None
        return out

    # ---- forward -------------------------------------------------------------------------------------------------
    @torch.compiler.disable
    def encode_image(self, x: torch.Tensor, normalize: bool = False) -> torch.Tensor:
        """x: float [B,3,H,W] normalised to [-1,1] (or uint8 [B,H,W,3]) -> [B,D] pooled embeddings; fp32, or the autocast
        dtype when called under torch.autocast (as open_clip's module would return)."""
        if self.weights_source == "random" and not self._warned_random:
            warnings.warn("dfd: this vision tower still carries seeded RANDOM weights - no pretrained checkpoint is "
                          "reachable offline and no backbone tensors were loaded; embeddings are meaningless until "
                          "load_state_dict() delivers `visual.trunk.*` (or `backbone.*`) tensors", stacklevel=2)
            self._warned_random = True
        self.sync_engine()
        out_dtype = torch.float32
        if torch.is_autocast_enabled("cuda"):
            out_dtype = torch.get_autocast_dtype("cuda")
        x = x.to(self._device, non_blocking=True)
        if x.dtype != torch.uint8 and x.dtype != torch.float32:
            x = x.float()
        mode = self.resize_mode & 0xF
        flip = self.resize_mode & ops.FLIP_H
        hw = x.shape[1:3] if x.dtype == torch.uint8 else x.shape[2:4]
        gp, P = self.arch.grid * self.arch.patch_size, self.arch.patch_size
        if not all(gp <= s < gp + P for s in hw) and mode == ops.RESIZE_NONE:
            mode = ops.RESIZE_BILINEAR
        with torch.cuda.device(self._device):
            pooled, _ = self.engine(x, resize_mode=mode | flip)
        f = pooled.float()
        if normalize:
            f = f / f.norm(dim=-1, keepdim=True)
        return f.to(out_dtype)

    def forward(self, image: torch.Tensor, text=None):
        if text is not None:
            raise NotImplementedError("dfd: only the vision tower of the SigLIP model is built (the reference never calls the text tower)")
        return self.encode_image(image)

    @property
    def device(self) -> torch.device:
        return self._device


def create_model_and_transforms(model_name: str, pretrained: Optional[str] = None, device="cuda", max_batch: int = 64,
                                state_dict: Optional[dict] = None, **_):
    """open_clip-shaped factory.  `pretrained` may be a local checkpoint path (.safetensors / .pt / .bin with open_clip
    or HF vision-tower keys); tags such as 'webli' cannot be resolved offline: the tower then keeps seeded random
    weights of the named architecture and says so (warning here, and once more on the first forward unless a
    checkpoint has been loaded through load_state_dict by then, which is what the reference scripts do next)."""
    if model_name not in ARCHS:
        raise KeyError(f"unknown model '{model_name}'; known: {sorted(ARCHS)}")
    arch = ARCHS[model_name]
    if state_dict is None and pretrained and os.path.exists(str(pretrained)):
        state_dict = _load_checkpoint_file(str(pretrained))
    elif state_dict is None and pretrained:
        warnings.warn(f"dfd: pretrained='{pretrained}' cannot be downloaded here; '{model_name}' starts from seeded random "
                      "weights until a checkpoint is loaded", stacklevel=2)
    model = VisionTower(arch, device, max_batch=max_batch, state_dict=state_dict)
    return model, None, make_preprocess(arch.image_size)


def _load_checkpoint_file(path: str) -> dict:
    if path.endswith(".safetensors"):
        from safetensors.torch import load_file

        return load_file(path)
    ck = torch.load(path, map_location="cpu", weights_only=True)
    for k in ("model_state_dict", "model_state", "state_dict", "model"):
        if isinstance(ck, dict) and k in ck and isinstance(ck[k], dict):
            return ck[k]
    return ck


class _Head:
    """Holder of classifier-head tensors with the reference's key names (classifier.N.*, se.N.*)."""

    def __init__(self, state: Dict[str, torch.Tensor], prefix: str):
        self.prefix = prefix
        self._state = state

    def state_dict(self):
        return {k[len(self.prefix):]: v for k, v in self._state.items() if k.startswith(self.prefix)}


class BinaryClassifier:
    """Both reference variants behind one class:
      head='A'  inference_ai_human_images.py:111-152 — f/||f||, LN -> Linear(D,D/2) -> GELU -> Linear(D/2,1)
      head='B'  train_fusion_head_only.py:78-109     — nearest resize if needed, f/(||f||+1e-6), SE gate, 3-layer MLP
    `model_size` follows the reference's tables; `arch` overrides it with any name in ARCHS."""

    SIZES = {"small": "ViT-B-16-SigLIP-384", "medium": "ViT-L-16-SigLIP-384", "large": "ViT-L-16-SigLIP-384",
             "so400m": "google/siglip2-so400m-patch14-384", "base224": "google/siglip2-base-patch16-224"}

    def __init__(self, model_size: str = "large", device="cuda", head: str = "A", arch: Optional[str] = None,
                 max_batch: int = 64, backbone_state: Optional[dict] = None, seed: int = 0):
        name = arch or self.SIZES[model_size]
        self.device = _as_device(device)
        self.backbone, _, self.preprocess = create_model_and_transforms(name, None, self.device, max_batch,
                                                                         backbone_state)
        self.arch = self.backbone.arch
        self.resolution = self.arch.image_size
        self.head_kind = head
        self._head_state = {k: v.clone() for k, v in random_classifier_head(head, self.arch.hidden_size, seed + 1).items()}
        self._params = None
        self.tta_flags = 0   # ops.FLIP_H: the forward reads every image mirrored (run_tta_inference's "H-Flip" pass)
        if head == "B":
            self.backbone.resize_mode = ops.RESIZE_NEAREST  # F.interpolate default (train_fusion_head_only.py:103-104)

    # reference attribute surface
    @property
    def classifier(self):
        return _Head(self._head_state, "classifier.")

    @property
    def se(self):
        return _Head(self._head_state, "se.")

    def eval(self):
        return self

    def train(self, mode: bool = True):
        return self

    def to(self, *a, **k):
        return self

    def parameters(self):
        return iter(())

    def state_dict(self):
        return dict(self._head_state)

    def load_state_dict(self, sd: dict, strict: bool = True):
        """Accepts the reference checkpoints (SURVEY.md App. B): `backbone.*` (+ ignored `backbone.text.*`) go to the
        engine, `classifier.*` / `se.*` to the head.  Non-strict loading drops shape mismatches like
        train_fusion_head_only.py:111-123."""
        sd = {k[len("_orig_mod."):] if k.startswith("_orig_mod.") else k: v for k, v in sd.items()}
        missing, unexpected = [], []
        for k in self._head_state:
            if k in sd and tuple(sd[k].shape) == tuple(self._head_state[k].shape):
                self._head_state[k] = sd[k].detach().float().cpu().clone()
            else:
                missing.append(k)
        bb = {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}
        if bb:
            r = self.backbone.load_state_dict(bb, strict=False)
            missing += ["backbone." + k for k in r.missing_keys]
            unexpected += ["backbone." + k for k in r.unexpected_keys]
        else:
            missing += ["backbone." + k for k, _ in self.backbone.named_parameters()]
        unexpected += [k for k in sd if not k.startswith("backbone.") and k not in self._head_state]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict: missing keys {missing[:8]}{'...' if len(missing) > 8 else ''}, "
                               f"unexpected keys {unexpected[:8]}{'...' if len(unexpected) > 8 else ''}")
        self._params = None
        return _IncompatibleKeys(missing, unexpected)

    def _head(self):
        if self._params is None:
            self._params = head_params_from_state(self._head_state, self.arch.hidden_size, self.device)
        return self._params

    def _pooled(self, x: torch.Tensor) -> torch.Tensor:
        x = x.to(self.device, non_blocking=True)
        if x.dtype not in (torch.uint8, torch.float32):
            x = x.float()
        hw = x.shape[1:3] if x.dtype == torch.uint8 else x.shape[2:4]
        mode = ops.RESIZE_NONE
        gp, P = self.arch.grid * self.arch.patch_size, self.arch.patch_size
        if not all(gp <= s < gp + P for s in hw):
            mode = (self.backbone.resize_mode & 0xF) or ops.RESIZE_BILINEAR
        self.backbone.sync_engine()
        with torch.cuda.device(self.device):
            return self.backbone.engine(x, resize_mode=mode | (self.tta_flags & ops.FLIP_H))[0]

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return ops.head_fwd(self._head(), self._pooled(x))[1]

    __call__ = forward

    def prototype_probs(self, x: torch.Tensor, prototypes: Dict[str, torch.Tensor]) -> torch.Tensor:
        """P(fake) = softmax([-||f-p_real||, -||f-p_fake||])[1]  (inference_ai_human_images.py:288-295), fused into the
        head kernel."""
        pr = torch.stack([prototypes["real"], prototypes["fake"]]).to(self.device, torch.float32).contiguous()
        return ops.head_fwd(self._head(), self._pooled(x), prototypes=pr)[2]

    def features(self, x: torch.Tensor) -> torch.Tensor:
        """L2-normalised embeddings f32 [B,D] (`encode_image` + `/ norm`)."""
        return ops.head_fwd(self._head(), self._pooled(x), want_features=True)[0]


class FastBinaryClassifier(BinaryClassifier):
    """cifake_binary_classifier.py:597-749 (BASELINE config 4): bilinear align_corners=False resize inside the model
    (32x32 CiFake images -> S), f/||f|| -> LayerNorm -> one-token attention -> size-dependent classifier (head H-D).
    State-dict keys follow the reference: layer_norm.*, attention.*, classifier.*."""

    CONFIGS = {"tiny": "ViT-B-16-SigLIP-256", "small": "ViT-B-16-SigLIP-384", "medium": "ViT-L-16-SigLIP-384",
               "large": "ViT-SO400M-16-SigLIP2-512"}

    def __init__(self, model_size: str = "small", device="cuda", arch: Optional[str] = None, max_batch: int = 64,
                 backbone_state: Optional[dict] = None, head_state: Optional[dict] = None, **_):
        name = arch or self.CONFIGS[model_size]
        self.model_size = model_size
        self.device = _as_device(device)
        self.backbone, _, self.preprocess = create_model_and_transforms(name, None, self.device, max_batch, backbone_state)
        self.arch = self.backbone.arch
        self.resolution = self.arch.image_size
        self.feature_dim = self.arch.hidden_size
        self.head_kind = "D"
        self.backbone.resize_mode = ops.RESIZE_BILINEAR
        self._head_state = {k: v.detach().float().cpu().clone() for k, v in (head_state or {}).items()}
        self._params = None
        self.tta_flags = 0

    def load_state_dict(self, sd: dict, strict: bool = True):
        sd = {k[len("_orig_mod."):] if k.startswith("_orig_mod.") else k: v for k, v in sd.items()}
        head = {k: v.detach().float().cpu().clone() for k, v in sd.items()
                if k.startswith(("layer_norm.", "attention.", "classifier."))}
        if head:
            self._head_state = head
        bb = {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}
        missing, unexpected = [], []
        if bb:
            r = self.backbone.load_state_dict(bb, strict=False)
            missing += ["backbone." + k for k in r.missing_keys]
            unexpected += ["backbone." + k for k in r.unexpected_keys]
        if strict and (not head or not bb or missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict: " + ("no head tensors; " if not head else "") +
                               ("no backbone.* tensors; " if not bb else "") + f"missing {missing[:8]} unexpected {unexpected[:8]}")
        self._params = None
        return _IncompatibleKeys(missing, unexpected)


def decode_only(pil) -> torch.Tensor:
    """Dataset transform for the device-side preprocess: the decoded pixels as a u8 [H,W,3] tensor, nothing else.  With
    `ragged_collate` the DataLoader workers only decode; `Resize((S,S))` (bit-exact PIL bilinear, dfd_resize_u8) runs on the GPU
    and ToTensor + Normalize(.5,.5) inside the patch kernel — inference_ai_human_images.py:200-204 without its host resize."""
    return torch.from_numpy(np.array(pil.convert("RGB"), dtype=np.uint8))


def ragged_collate(batch):
    """collate_fn for `decode_only` samples: images of different sizes stay a list; labels / filenames as the default collate."""
    imgs, labels, names = zip(*batch)
    return list(imgs), torch.as_tensor(labels), list(names)


def resize_on_device(model: "BinaryClassifier", images) -> torch.Tensor:
    """A ragged list of u8 [H,W,3] host tensors -> u8 [B,S,S,3] on the model's device: one upload per image at its decoded size,
    PIL-exact bilinear resize there (images that already are SxS are taken as they are, like PIL's no-op resize)."""
    S = model.resolution
    out = []
    with torch.cuda.device(model.device):
        for im in images:
            d = im.to(model.device, non_blocking=True)[None]
            out.append(d if tuple(d.shape[1:3]) == (S, S) else ops.resize_u8(d, S, S, "bilinear"))
        return torch.cat(out)


@torch.no_grad()
def run_inference(model: BinaryClassifier, dataloader, device=None, use_amp: bool = True, desc: str = "Inference",
                  invert_logits: bool = False, prototypes: Optional[dict] = None):
    """inference_ai_human_images.py:250-318: loader of (images, labels, filenames) -> (labels, P(fake), filenames).
    One D2H read per batch, like the reference loop.  `images` is either the reference's normalised float batch [B,3,S,S] or,
    from a `decode_only` / `ragged_collate` loader, a list of decoded u8 images that are resized on the device."""
    all_labels, all_probs, all_files = [], [], []
    for images, labels, filenames in dataloader:
        if isinstance(images, (list, tuple)):
            images = resize_on_device(model, images)
        if prototypes is not None:
            probs = model.prototype_probs(images, prototypes)
        else:
            z = model(images)
            probs = torch.sigmoid(-z if invert_logits else z)
        all_probs.extend(probs.cpu().numpy())
        all_labels.extend(np.asarray(labels))
        all_files.extend(filenames)
    return np.array(all_labels), np.array(all_probs), all_files


class AIHumanDataset(torch.utils.data.Dataset):
    """(image, label, filename) triples from a metadata CSV with `file_name` (path relative to data_dir) and `label`
    (0 real / 1 fake) columns - inference_ai_human_images.py:155-192.  Rows whose file does not exist are dropped."""

    def __init__(self, data_dir, metadata_csv, transform=None, max_samples: Optional[int] = None):
        import pandas as pd

        self.transform = transform
        df = pd.read_csv(metadata_csv)
        self.samples = [(os.path.join(str(data_dir), str(f)), int(lab), str(f))
                        for f, lab in zip(df["file_name"], df["label"]) if os.path.exists(os.path.join(str(data_dir), str(f)))]
        if max_samples and len(self.samples) > max_samples:
            keep = np.random.choice(len(self.samples), max_samples, replace=False)
            self.samples = [self.samples[i] for i in keep]

    def __len__(self):
        return len(self.samples)

    def __getitem__(self, i):
        from PIL import Image

        path, label, name = self.samples[i]
        try:
            img = Image.open(path).convert("RGB")
        except Exception:   # unreadable file -> black image, as the reference's loader does (:77-80)
            img = Image.new("RGB", (384, 384), color="black")
        return (self.transform(img) if self.transform else img), label, name


def _clahe_lab(pil):
    """CLAHE(2.0, 8x8) on the L channel of LAB (inference_ai_human_images.py:83-97)."""
    import cv2
    from PIL import Image

    img = np.array(pil)
    cl = cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8, 8))
    if img.ndim == 3:
        lab = cv2.cvtColor(img, cv2.COLOR_RGB2LAB)
        lab[:, :, 0] = cl.apply(lab[:, :, 0])
        img = cv2.cvtColor(lab, cv2.COLOR_LAB2RGB)
    else:
        img = cl.apply(img)
    return Image.fromarray(img)


def _sharpen(pil):
    """ImageFilter.SHARPEN then Sharpness x1.5 (inference_ai_human_images.py:100-108)."""
    from PIL import ImageEnhance, ImageFilter

    return ImageEnhance.Sharpness(pil.filter(ImageFilter.SHARPEN)).enhance(1.5)


TTA_NAMES = ("Original", "H-Flip", "CLAHE", "Sharpen", "CLAHE+Sharpen")


def create_tta_transforms(image_size: int, num_augments: int = 5):
    """[(name, transform)] in the reference's order (inference_ai_human_images.py:195-247): Resize((S,S)) [+ H-flip |
    CLAHE | sharpen | both] + ToTensor + Normalize(.5,.5).  Host-side PIL transforms, exactly like the reference; the
    first two are also available without a second decode/upload through `run_tta_inference` (DFD_FLIP_H pass)."""
    from torchvision import transforms

    def make(extra):
        return transforms.Compose([transforms.Resize((image_size, image_size))] + extra +
                                  [transforms.ToTensor(), transforms.Normalize([0.5] * 3, [0.5] * 3)])

    extras = [[], [transforms.RandomHorizontalFlip(p=1.0)], [transforms.Lambda(_clahe_lab)], [transforms.Lambda(_sharpen)],
              [transforms.Lambda(lambda im: _sharpen(_clahe_lab(im)))]]
    return [(TTA_NAMES[i], make(extras[i])) for i in range(max(1, min(num_augments, 5)))]


def run_tta_inference(model, data_dir, metadata_csv, tta_transforms, batch_size, num_workers=0, device=None,
                      use_amp: bool = True, invert_logits: bool = False, prototypes: Optional[dict] = None,
                      device_resize: bool = False):
    """inference_ai_human_images.py:321-360: one pass per TTA transform, probabilities averaged.
    Returns (y_true, mean probabilities, [per-transform probabilities], filenames).

    The reference decodes, resizes and uploads the dataset once per transform.  For the default configuration
    (NUM_TTA_AUGMENTS = 2: "Original" + "H-Flip", :731-732) and a dfd BinaryClassifier the mirrored view is produced by
    the patch kernel from the pixels that are already resident (DFD_FLIP_H), so both views cost one decode and one
    upload per image; the remaining transforms (CLAHE / sharpen, host PIL ops in the reference too) run as extra passes.
    device_resize: the fused "Original" + "H-Flip" pass decodes on the host only (`decode_only` + `ragged_collate`) and does the
    `Resize((S,S))` on the GPU as well (bit-exact with PIL, see `resize_on_device`)."""
    from torch.utils.data import DataLoader

    names = [n for n, _ in tta_transforms]
    fused = (isinstance(model, BinaryClassifier) and len(names) >= 2 and names[0] == "Original" and names[1] == "H-Flip")
    all_probs, y_true, filenames = [], None, None

    def loader(tf, ragged=False):
        ds = AIHumanDataset(data_dir, metadata_csv, transform=tf)
        return DataLoader(ds, batch_size=batch_size, shuffle=False, num_workers=num_workers,
                          pin_memory=torch.cuda.is_available() and not ragged, persistent_workers=False,
                          collate_fn=ragged_collate if ragged else None)

    start = 0
    if fused:
        labs, p0, p1, files = [], [], [], []
        with torch.no_grad():
            for images, labels, fn in (loader(decode_only, True) if device_resize else loader(tta_transforms[0][1])):
                images = resize_on_device(model, images) if device_resize else images.to(model.device, non_blocking=True)
                for flags, acc in ((0, p0), (ops.FLIP_H, p1)):
                    model.tta_flags = flags
                    try:
                        if prototypes is not None:
                            pr = model.prototype_probs(images, prototypes)
                        else:
                            z = model(images)
                            pr = torch.sigmoid(-z if invert_logits else z)
                    finally:
                        model.tta_flags = 0
                    acc.extend(pr.cpu().numpy())
                labs.extend(np.asarray(labels))
                files.extend(fn)
        y_true, filenames = np.array(labs), files
        all_probs += [np.array(p0), np.array(p1)]
        start = 2
    for name, tf in tta_transforms[start:]:
        labels, probs, fnames = run_inference(model, loader(tf), device, use_amp, desc=f"  {name}",
                                              invert_logits=invert_logits, prototypes=prototypes)
        if y_true is None:
            y_true, filenames = labels, fnames
        else:
            assert np.array_equal(y_true, labels), "Labels mismatch across TTA!"
        all_probs.append(probs)
    return y_true, np.mean(all_probs, axis=0), all_probs, filenames


@torch.no_grad()
def few_shot_prototype(model: BinaryClassifier, support_loader, device=None, use_amp: bool = True) -> dict:
    """inference_ai_human_images.py:477-541: L2-normalised class means of L2-normalised features.  Class sums are
    accumulated on the device; with torch.distributed initialised they are all-reduced so every rank gets the
    same prototypes (SURVEY.md §8e)."""
    from . import distributed

    D = model.arch.hidden_size
    sums = torch.zeros(2, D, device=model.device)
    counts = torch.zeros(2, device=model.device)
    for images, labels, _ in support_loader:
        f = model.features(images)
        lab = (torch.as_tensor(labels).to(model.device) != 0).long()
        sums.index_add_(0, lab, f)
        counts.index_add_(0, lab, torch.ones_like(lab, dtype=torch.float32))
    bucket = torch.cat([sums.reshape(-1), counts])
    distributed.all_reduce_sum_(bucket)
    sums, counts = bucket[: 2 * D].reshape(2, D), bucket[2 * D:]
    means = sums / counts.clamp_min(1.0)[:, None]
    protos = means / means.norm(dim=-1, keepdim=True)
    return {"real": protos[0], "fake": protos[1]}


def interpolated_position_table(pos: torch.Tensor, new_grid: int) -> torch.Tensor:
    """HF `SiglipVisionEmbeddings.interpolate_pos_encoding` (HF:modeling_siglip.py:137-173) for a square grid:
    [N,D] table viewed as [1,D,G,G], bicubic (align_corners=False, no antialias) to new_grid x new_grid, back to [N',D].
    Done once per grid size when the engine for that size is created (a load-time step, like the weight repack)."""
    N, D = pos.shape
    G = int(round(N ** 0.5))
    if G * G != N:
        raise ValueError("position table is not a square grid")
    t = pos.detach().float().reshape(1, G, G, D).permute(0, 3, 1, 2)
    t = torch.nn.functional.interpolate(t, size=(new_grid, new_grid), mode="bicubic", align_corners=False)
    return t.permute(0, 2, 3, 1).reshape(new_grid * new_grid, D).contiguous()


class SiglipVisionModel:
    """HF-shaped wrapper: `SiglipVisionModel.from_state_dict(sd)(pixel_values=x)` -> .pooler_output [B,D] f32,
    .last_hidden_state [B,N,D], and with output_hidden_states=True the tuple of L+1 per-layer states
    (Siglip2sidafrozen.py:753,787-793).  output_attentions=True adds .attentions, the tuple of L fp32 [B,H,N,N]
    attention probabilities that HF returns under eager attention (None otherwise).  `interpolate_pos_encoding=True` (Siglip2sidafrozen.py:787, progressive resize
    :975-987) accepts other square resolutions: each new patch grid gets its own engine (workspace sized for that token
    count) whose position table is the bicubic resample of the trained one."""

    def __init__(self, arch: VisionArch, state_dict: dict, device="cuda", max_batch: int = 32):
        self.arch = arch
        self.device = _as_device(device)
        self.max_batch = max_batch
        self.config = types.SimpleNamespace(hidden_size=arch.hidden_size, image_size=arch.image_size,
                                            patch_size=arch.patch_size, num_hidden_layers=arch.num_hidden_layers,
                                            num_attention_heads=arch.num_attention_heads,
                                            intermediate_size=arch.intermediate_size)
        self._canon = canonicalize_state_dict(state_dict)
        self.engine = SiglipEngine(arch, self.device.index, max_batch).load_state_dict(self._canon)
        self._engines = {arch.grid: self.engine}

    @classmethod
    def from_state_dict(cls, state_dict: dict, device="cuda", max_batch: int = 32, num_heads: Optional[int] = None):
        return cls(arch_from_state_dict(state_dict, num_heads), state_dict, device, max_batch)

    def eval(self):
        return self

    def to(self, *a, **k):
        return self

    def engine_for_grid(self, grid: int) -> SiglipEngine:
        if grid not in self._engines:
            a = self.arch
            arch = VisionArch(grid * a.patch_size, a.patch_size, a.hidden_size, a.intermediate_size, a.num_hidden_layers,
                              a.num_attention_heads, a.layer_norm_eps)
            sd = dict(self._canon)
            sd["embeddings.position_embedding.weight"] = interpolated_position_table(
                self._canon["embeddings.position_embedding.weight"], grid)
            # keep the activation workspace of the extra engine in proportion to the native one's
            mb = max(1, min(self.max_batch, self.max_batch * a.tokens // (grid * grid)))
            self._engines[grid] = SiglipEngine(arch, self.device.index, mb).load_state_dict(sd)
        return self._engines[grid]

    def __call__(self, pixel_values: torch.Tensor, output_hidden_states: bool = False,
                 interpolate_pos_encoding: bool = False, output_attentions: bool = False, **_):
        P = self.arch.patch_size
        H, W = pixel_values.shape[-2:]
        gh, gw = H // P, W // P
        if (gh, gw) == (self.arch.grid, self.arch.grid):
            eng = self.engine
        elif interpolate_pos_encoding and gh == gw and gh >= 1:
            eng = self.engine_for_grid(gh)
        elif not interpolate_pos_encoding:
            raise ValueError(f"pixel_values of {H}x{W} give a {gh}x{gw} patch grid, the model has {self.arch.grid}x"
                             f"{self.arch.grid}; pass interpolate_pos_encoding=True (as HF requires)")
        else:
            raise NotImplementedError("interpolate_pos_encoding for non-square inputs is not built (the reference's "
                                      "SigLIP2_MTL needs square token grids too: Siglip2sidafrozen.py:795-801)")
        x = pixel_values.to(self.device).float()
        if output_attentions:  # HF eager: a tuple of L fp32 [B,H,N,N]; one engine forward per chunk gives every output
            chunks = [eng._forward_tapped(x[i:i + eng.max_batch], 0, True, output_hidden_states, True)
                      for i in range(0, x.shape[0], eng.max_batch)]
            pooled = torch.cat([c[0] for c in chunks])
            last = torch.cat([c[1] for c in chunks])
            attn = torch.cat([c[2] for c in chunks], 1)
            hid = tuple(h.float() for h in torch.cat([c[4] for c in chunks], 1)) if output_hidden_states else None
            return types.SimpleNamespace(pooler_output=pooled.float(), last_hidden_state=last.float(), hidden_states=hid,
                                         attentions=tuple(attn.unbind(0)))
        if output_hidden_states:  # tuple of L+1 tensors, as SigLIP2_MTL consumes them (Siglip2sidafrozen.py:790-793)
            chunks = [eng.forward_hidden(x[i:i + eng.max_batch]) for i in range(0, x.shape[0], eng.max_batch)]
            pooled = torch.cat([c[0] for c in chunks])
            last = torch.cat([c[1] for c in chunks])
            hid = torch.cat([c[2] for c in chunks], 1)
            return types.SimpleNamespace(pooler_output=pooled.float(), last_hidden_state=last.float(),
                                         hidden_states=tuple(h.float() for h in hid), attentions=None)
        pooled, last = eng(x, want_last_hidden=True)
        return types.SimpleNamespace(pooler_output=pooled.float(), last_hidden_state=last.float(), hidden_states=None,
                                     attentions=None)


def install_import_shims() -> None:
    """Make `import open_clip` / `import pywt` resolve to dfd-backed stand-ins (the reference scripts import both at
    module level; neither package is installed here)."""
    oc = types.ModuleType("open_clip")
    oc.create_model_and_transforms = create_model_and_transforms
    oc.__doc__ = "dfd stand-in for open_clip (vision tower only)"
    sys.modules.setdefault("open_clip", oc)

    pw = types.ModuleType("pywt")

    def dwt2(x, wavelet):
        if wavelet not in ("db1", "haar"):
            raise ValueError("dfd pywt stand-in only implements the db1 / Haar wavelet")
        a = np.asarray(x)
        p, q, r, s = a[0::2, 0::2], a[0::2, 1::2], a[1::2, 0::2], a[1::2, 1::2]
        return (p + q + r + s) * 0.5, ((p + q - r - s) * 0.5, (p - q + r - s) * 0.5, (p - q - r + s) * 0.5)

    pw.dwt2 = dwt2
    sys.modules.setdefault("pywt", pw)

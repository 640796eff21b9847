"""ORACLE (test infrastructure, not product code) — CPU restatement of the SigLIP vision tower forward.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.

The arithmetic lives in a third-party dependency of the reference that is NOT under /root/reference:
HuggingFace `transformers` (unpinned by the reference; 5.5.0 in this image), called by the reference at
Siglip2sidafrozen.py:52,753,787-788.  This file restates transformers/models/siglip/modeling_siglip.py
("HF:" below) in plain fp32 torch-on-CPU tensor algebra:

  embeddings      HF:124-135,175-186   conv k=s=P, padding valid -> flatten -> + position embedding
  encoder layer   HF:340-362           pre-LN block, eps 1e-6
  attention       HF:229-249,275-312   softmax(q k^T / sqrt(hd)) v, non causal, fp32 softmax
  mlp             HF:315-327           fc1 -> gelu_pytorch_tanh -> fc2
  tail            HF:586-625           post_layernorm
  MAP head        HF:628-654           probe query, nn.MultiheadAttention (packed in_proj), LN, MLP residual

Pinned: oracle/make_golden.py runs the real `transformers.SiglipVisionModel` on the same weights/inputs
and tests/test_oracle_cpu.py checks this restatement against those committed outputs (tests/golden/).

mode="fp32"      exact fp32 everywhere (the mathematical reference)
mode="autocast"  rounds where torch.autocast(bfloat16) rounds: GEMM operands and outputs and SDPA in bf16,
                 LayerNorm / softmax / residual stream in fp32 — the "reference PyTorch/HF path in bf16"
                 of BASELINE.json, reproducible without a GPU.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F


@dataclass(frozen=True)
class VisionConfig:
    image_size: int
    patch_size: int
    hidden_size: int
    intermediate_size: int
    num_hidden_layers: int
    num_attention_heads: int
    layer_norm_eps: float = 1e-6

    @property
    def grid(self):
        return self.image_size // self.patch_size

    @property
    def tokens(self):
        return self.grid * self.grid

    @property
    def head_dim(self):
        return self.hidden_size // self.num_attention_heads


CONFIGS = {
    # SURVEY.md App. C
    "siglip2-base-patch16-224": VisionConfig(224, 16, 768, 3072, 12, 12),
    "siglip2-so400m-patch14-384": VisionConfig(384, 14, 1152, 4304, 27, 16),
    "siglip2-large-patch16-384": VisionConfig(384, 16, 1024, 4096, 24, 16),
    # small shapes for parity tests: hd=64 / hd=72, ragged N, inter not a multiple of 64
    "tiny-hd64": VisionConfig(64, 16, 128, 256, 2, 2),
    "tiny-hd72": VisionConfig(60, 14, 144, 304, 2, 2),
    "small-hd72": VisionConfig(210, 14, 288, 1080, 3, 4),
}


def flops_per_image(c: VisionConfig) -> float:
    """Algorithmic FLOPs of one forward (SURVEY.md §8d): 2MNK per GEMM, 4N²D per attention layer."""
    N, D, I, L, P = c.tokens, c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.patch_size
    pe = 2 * N * 3 * P * P * D
    layer = 8 * N * D * D + 4 * N * D * I + 4 * N * N * D
    mp = 4 * N * D * D + 4 * D * D + 4 * N * D + 4 * D * I
    return float(pe + L * layer + mp)


def init_state_dict(c: VisionConfig, seed: int = 0) -> dict:
    """Seeded random weights in the HF key layout (without the 'vision_model.' prefix).  Gains are chosen so
    attention logits, GELU inputs and biases are all O(1) — a wrong kernel cannot hide behind tiny values."""
    g = torch.Generator().manual_seed(seed)
    D, I, P, N = c.hidden_size, c.intermediate_size, c.patch_size, c.tokens

    def rn(*shape, std=1.0):
        return torch.randn(*shape, generator=g, dtype=torch.float32) * std

    def lin(prefix, out_f, in_f, sd, gain=1.0):
        sd[prefix + ".weight"] = rn(out_f, in_f, std=gain / math.sqrt(in_f))
        sd[prefix + ".bias"] = rn(out_f, std=0.1)

    def ln(prefix, sd):
        sd[prefix + ".weight"] = 1.0 + rn(D, std=0.1)
        sd[prefix + ".bias"] = rn(D, std=0.1)

    sd = {}
    sd["embeddings.patch_embedding.weight"] = rn(D, 3, P, P, std=1.0 / math.sqrt(3 * P * P))
    sd["embeddings.patch_embedding.bias"] = rn(D, std=0.1)
    sd["embeddings.position_embedding.weight"] = rn(N, D, std=0.5)
    for i in range(c.num_hidden_layers):
        p = f"encoder.layers.{i}"
        ln(p + ".layer_norm1", sd)
        ln(p + ".layer_norm2", sd)
        for nm in ("q_proj", "k_proj", "v_proj"):
            lin(f"{p}.self_attn.{nm}", D, D, sd, gain=1.5 if nm != "v_proj" else 1.0)
        lin(f"{p}.self_attn.out_proj", D, D, sd, gain=0.5)
        lin(f"{p}.mlp.fc1", I, D, sd)
        lin(f"{p}.mlp.fc2", D, I, sd, gain=0.5)
    ln("post_layernorm", sd)
    sd["head.probe"] = rn(1, 1, D)
    sd["head.attention.in_proj_weight"] = rn(3 * D, D, std=1.5 / math.sqrt(D))
    sd["head.attention.in_proj_bias"] = rn(3 * D, std=0.1)
    lin("head.attention.out_proj", D, D, sd)
    ln("head.layernorm", sd)
    lin("head.mlp.fc1", I, D, sd)
    lin("head.mlp.fc2", D, I, sd, gain=0.5)
    return sd


def synthetic_images(B: int, S: int, seed: int = 0) -> torch.Tensor:
    """uint8 NHWC images, SURVEY.md §8d."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, generator=g)


def preprocess_u8(img_u8_nhwc: torch.Tensor) -> torch.Tensor:
    """ToTensor + Normalize(.5,.5) (inference_ai_human_images.py:200-204): u8 NHWC -> f32 NCHW in [-1,1]."""
    x = img_u8_nhwc.permute(0, 3, 1, 2).to(torch.float32) / 255.0
    return (x - 0.5) / 0.5


def resize_input(x: torch.Tensor, S: int, mode: str) -> torch.Tensor:
    """In-model resample of the normalised tensor: 'nearest' (train_fusion_head_only.py:103-104),
    'bilinear' align_corners=False (cifake_binary_classifier.py:716-717)."""
    if x.shape[-1] == S and x.shape[-2] == S:
        return x
    if mode == "nearest":
        return F.interpolate(x, size=(S, S))
    if mode == "bilinear":
        return F.interpolate(x, size=(S, S), mode="bilinear", align_corners=False)
    raise ValueError(mode)


def _rb(t: torch.Tensor, on: bool) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float32) if on else t


def _linear(x, w, b, ac):
    y = _rb(x, ac) @ _rb(w, ac).t() + (_rb(b, ac) if b is not None else 0.0)
    return _rb(y, ac)


def _layernorm(x, g, b, eps):
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * g + b


def _gelu_tanh(x):
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


def _mha(q, k, v, H, ac, scale=None):
    """q [B,Nq,D], k/v [B,Nk,D] -> [B,Nq,D]; softmax in fp32; P and the output round to bf16 under autocast.
    scale: the logit scale, 1/sqrt(head dim) unless given."""
    B, Nq, D = q.shape
    hd = D // H
    qh = _rb(q, ac).view(B, Nq, H, hd).transpose(1, 2)
    kh = _rb(k, ac).view(B, -1, H, hd).transpose(1, 2)
    vh = _rb(v, ac).view(B, -1, H, hd).transpose(1, 2)
    s = (qh @ kh.transpose(-1, -2)) * (hd ** -0.5 if scale is None else scale)
    p = torch.softmax(s, dim=-1)
    o = _rb(p, ac) @ vh
    return _rb(o.transpose(1, 2).reshape(B, Nq, D), ac)


def _check_mode(mode: str) -> bool:
    assert mode in ("fp32", "autocast")
    return mode == "autocast"


# The three stages below compute in the dtype of their inputs (float32, or float64 with a float64 state dict),
# so mode="fp32" on float64 tensors is a float64 reference of the same arithmetic.
@torch.no_grad()
def embed(sd: dict, c: VisionConfig, pixel_values: torch.Tensor, mode: str = "fp32") -> torch.Tensor:
    """pixel_values [B,3,S,S] (already normalised) -> hidden_states[0] [B,N,D]: patch embedding + position."""
    ac = _check_mode(mode)
    B = pixel_values.shape[0]
    P, G, D = c.patch_size, c.grid, c.hidden_size
    # conv k=s=P, padding valid == im2col over the top-left G*P x G*P crop, column order (c, ky, kx)
    x = pixel_values[:, :, : G * P, : G * P]
    if x.dtype != torch.float64:
        x = x.to(torch.float32)
    patches = x.reshape(B, 3, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(B, G * G, 3 * P * P)
    w = sd["embeddings.patch_embedding.weight"].reshape(D, -1)
    h = _linear(patches, w, sd["embeddings.patch_embedding.bias"], ac)
    return h + sd["embeddings.position_embedding.weight"][None]


@torch.no_grad()
def encoder_layer(sd: dict, c: VisionConfig, i: int, h: torch.Tensor, mode: str = "fp32",
                  attn_scale: float | None = None) -> torch.Tensor:
    """hidden_states[i] [B,N,D] -> hidden_states[i+1]: encoder layer i (pre-LN attention block, then pre-LN MLP).
    attn_scale overrides the attention logit scale 1/sqrt(head dim) (tests use it to measure a kernel's effective scale)."""
    ac = _check_mode(mode)
    eps = c.layer_norm_eps
    p = f"encoder.layers.{i}."
    y = _layernorm(h, sd[p + "layer_norm1.weight"], sd[p + "layer_norm1.bias"], eps)
    q = _linear(y, sd[p + "self_attn.q_proj.weight"], sd[p + "self_attn.q_proj.bias"], ac)
    k = _linear(y, sd[p + "self_attn.k_proj.weight"], sd[p + "self_attn.k_proj.bias"], ac)
    v = _linear(y, sd[p + "self_attn.v_proj.weight"], sd[p + "self_attn.v_proj.bias"], ac)
    a = _mha(q, k, v, c.num_attention_heads, ac, attn_scale)
    h = h + _linear(a, sd[p + "self_attn.out_proj.weight"], sd[p + "self_attn.out_proj.bias"], ac)
    y = _layernorm(h, sd[p + "layer_norm2.weight"], sd[p + "layer_norm2.bias"], eps)
    m = _rb(_gelu_tanh(_linear(y, sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"], ac)), ac)
    return h + _linear(m, sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"], ac)


@torch.no_grad()
def post_layernorm(sd: dict, c: VisionConfig, h: torch.Tensor) -> torch.Tensor:
    """hidden_states[L] -> last_hidden_state."""
    return _layernorm(h, sd["post_layernorm.weight"], sd["post_layernorm.bias"], c.layer_norm_eps)


@torch.no_grad()
def map_head(sd: dict, c: VisionConfig, last: torch.Tensor, mode: str = "fp32") -> torch.Tensor:
    """last_hidden_state [B,N,D] -> pooler_output [B,D]: MAP pooling (probe attention, LayerNorm, MLP residual)."""
    ac = _check_mode(mode)
    B, D = last.shape[0], c.hidden_size
    wi, bi = sd["head.attention.in_proj_weight"], sd["head.attention.in_proj_bias"]
    probe = sd["head.probe"].reshape(1, 1, D).expand(B, 1, D)
    q = _linear(probe, wi[:D], bi[:D], ac)
    k = _linear(last, wi[D : 2 * D], bi[D : 2 * D], ac)
    v = _linear(last, wi[2 * D :], bi[2 * D :], ac)
    a = _mha(q, k, v, c.num_attention_heads, ac)
    r = _linear(a, sd["head.attention.out_proj.weight"], sd["head.attention.out_proj.bias"], ac)
    y = _layernorm(r, sd["head.layernorm.weight"], sd["head.layernorm.bias"], c.layer_norm_eps)
    m = _rb(_gelu_tanh(_linear(y, sd["head.mlp.fc1.weight"], sd["head.mlp.fc1.bias"], ac)), ac)
    out = r + _linear(m, sd["head.mlp.fc2.weight"], sd["head.mlp.fc2.bias"], ac)
    return out[:, 0]


@torch.no_grad()
def siglip_vision_forward(sd: dict, c: VisionConfig, pixel_values: torch.Tensor, mode: str = "fp32",
                          output_hidden_states: bool = False) -> dict:
    """pixel_values f32 [B,3,S,S] (already normalised) -> {'pooler_output' [B,D], 'last_hidden_state' [B,N,D],
    'hidden_states' tuple of L+1 (optional)}."""
    h = embed(sd, c, pixel_values, mode)
    hidden = [h]
    for i in range(c.num_hidden_layers):
        h = encoder_layer(sd, c, i, h, mode)
        hidden.append(h)
    last = post_layernorm(sd, c, h)
    res = {"pooler_output": map_head(sd, c, last, mode), "last_hidden_state": last}
    if output_hidden_states:
        res["hidden_states"] = tuple(hidden)
    return res


# ---- classifier heads on pooled embeddings --------------------------------------------------------------
def l2_normalize(f: torch.Tensor, eps: float = 0.0) -> torch.Tensor:
    """inference_ai_human_images.py:149 (eps 0) / train_fusion_head_only.py:106 (eps 1e-6)."""
    return f / (f.norm(dim=-1, keepdim=True) + eps)


def init_head(kind: str, D: int, seed: int = 1) -> dict:
    g = torch.Generator().manual_seed(seed)

    def rn(*shape, std):
        return torch.randn(*shape, generator=g, dtype=torch.float32) * std

    sd = {}
    if kind == "B":
        sd["se.0.weight"], sd["se.0.bias"] = rn(D // 16, D, std=2.0), rn(D // 16, std=0.1)
        sd["se.2.weight"], sd["se.2.bias"] = rn(D, D // 16, std=1.0 / math.sqrt(D // 16)), rn(D, std=0.1)
    sd["classifier.0.weight"], sd["classifier.0.bias"] = 1.0 + rn(D, std=0.1), rn(D, std=0.1)
    sd["classifier.2.weight"], sd["classifier.2.bias"] = rn(D // 2, D, std=1.0 / math.sqrt(D)), rn(D // 2, std=0.1)
    if kind == "A":
        sd["classifier.5.weight"], sd["classifier.5.bias"] = rn(1, D // 2, std=1.0 / math.sqrt(D // 2)), rn(1, std=0.1)
    else:
        sd["classifier.5.weight"] = rn(D // 4, D // 2, std=1.0 / math.sqrt(D // 2))
        sd["classifier.5.bias"] = rn(D // 4, std=0.1)
        sd["classifier.7.weight"], sd["classifier.7.bias"] = rn(1, D // 4, std=1.0 / math.sqrt(D // 4)), rn(1, std=0.1)
    return sd


@torch.no_grad()
def classifier_head(sd: dict, kind: str, pooled: torch.Tensor, norm_eps: float) -> torch.Tensor:
    """H-A: inference_ai_human_images.py:131-138,148-152.  H-B: train_fusion_head_only.py:84-99,105-108.
    Dropout is identity in eval.  GELU is exact erf."""
    f = l2_normalize(pooled.to(torch.float32), norm_eps)
    if kind == "B":
        se = torch.sigmoid(torch.relu(f @ sd["se.0.weight"].t() + sd["se.0.bias"]) @ sd["se.2.weight"].t()
                           + sd["se.2.bias"])
        f = f * se
    y = F.layer_norm(f, (f.shape[-1],), sd["classifier.0.weight"], sd["classifier.0.bias"], 1e-5)
    y = F.gelu(y @ sd["classifier.2.weight"].t() + sd["classifier.2.bias"])
    if kind == "A":
        return (y @ sd["classifier.5.weight"].t() + sd["classifier.5.bias"]).squeeze(-1)
    y = F.gelu(y @ sd["classifier.5.weight"].t() + sd["classifier.5.bias"])
    return (y @ sd["classifier.7.weight"].t() + sd["classifier.7.bias"]).squeeze(-1)


def init_head_d(model_size: str, D: int, seed: int = 4) -> dict:
    """FastBinaryClassifier head state dict (cifake_binary_classifier.py:643-687): layer_norm, attention
    (LightweightAttention for tiny/small, nn.MultiheadAttention for large, none for medium), classifier."""
    g = torch.Generator().manual_seed(seed)

    def rn(*shape, std):
        return torch.randn(*shape, generator=g, dtype=torch.float32) * std

    sd = {"layer_norm.weight": 1.0 + rn(D, std=0.1), "layer_norm.bias": rn(D, std=0.1)}
    if model_size in ("tiny", "small"):
        sd["attention.qkv.weight"], sd["attention.qkv.bias"] = rn(3 * D, D, std=1.0 / math.sqrt(D)), rn(3 * D, std=0.1)
        sd["attention.proj.weight"], sd["attention.proj.bias"] = rn(D, D, std=1.0 / math.sqrt(D)), rn(D, std=0.1)
    elif model_size == "large":
        sd["attention.in_proj_weight"], sd["attention.in_proj_bias"] = rn(3 * D, D, std=1.0 / math.sqrt(D)), rn(3 * D, std=0.1)
        sd["attention.out_proj.weight"], sd["attention.out_proj.bias"] = rn(D, D, std=1.0 / math.sqrt(D)), rn(D, std=0.1)
    if model_size == "tiny":
        dims, idx = [D, 1], [1]
    elif model_size == "small":
        dims, idx = [D, D // 4, 1], [0, 3]
    else:
        dims, idx = [D, D // 2, D // 4, 1], [0, 3, 6]
    for i, n in enumerate(idx):
        sd[f"classifier.{n}.weight"] = rn(dims[i + 1], dims[i], std=1.0 / math.sqrt(dims[i]))
        sd[f"classifier.{n}.bias"] = rn(dims[i + 1], std=0.1)
    return sd


@torch.no_grad()
def classifier_head_d(sd: dict, pooled: torch.Tensor) -> torch.Tensor:
    """cifake_binary_classifier.py:727-749: f/||f|| -> LayerNorm -> attention over ONE token -> classifier.
    With a single token the softmax weight is exactly 1, so attention(x) = proj(v(x))."""
    f = l2_normalize(pooled.to(torch.float32), 0.0)
    D = f.shape[-1]
    y = F.layer_norm(f, (D,), sd["layer_norm.weight"], sd["layer_norm.bias"], 1e-5)
    if "attention.qkv.weight" in sd:
        v = y @ sd["attention.qkv.weight"][2 * D:].t() + sd["attention.qkv.bias"][2 * D:]
        y = v @ sd["attention.proj.weight"].t() + sd["attention.proj.bias"]
    elif "attention.in_proj_weight" in sd:
        v = y @ sd["attention.in_proj_weight"][2 * D:].t() + sd["attention.in_proj_bias"][2 * D:]
        y = v @ sd["attention.out_proj.weight"].t() + sd["attention.out_proj.bias"]
    idx = sorted(int(k.split(".")[1]) for k in sd if k.startswith("classifier.") and k.endswith(".weight"))
    for n, i in enumerate(idx):
        y = y @ sd[f"classifier.{i}.weight"].t() + sd[f"classifier.{i}.bias"]
        if n + 1 < len(idx):
            y = F.gelu(y)
    return y.squeeze(-1)


@torch.no_grad()
def prototype_prob(features: torch.Tensor, real_proto: torch.Tensor, fake_proto: torch.Tensor) -> torch.Tensor:
    """inference_ai_human_images.py:288-295: softmax([-d_real, -d_fake])[:, 1] with Euclidean cdist."""
    dr = torch.cdist(features, real_proto[None])
    df = torch.cdist(features, fake_proto[None])
    return torch.softmax(torch.cat([-dr, -df], dim=1), dim=1)[:, 1]


def cosine_report(a: torch.Tensor, b: torch.Tensor) -> dict:
    """Cosine per row, also after removing the batch-mean embedding (SURVEY.md §8d caveat), and rel-L2."""
    a, b = a.to(torch.float64), b.to(torch.float64)
    cos = F.cosine_similarity(a, b, dim=-1)
    out = {"cos_min": float(cos.min()), "rel_l2": float((a - b).norm() / b.norm())}
    if a.shape[0] > 1:
        ac, bc = a - b.mean(0, keepdim=True), b - b.mean(0, keepdim=True)
        out["cos_centered_min"] = float(F.cosine_similarity(ac, bc, dim=-1).min())
    return out

"""Reference attention maps for the tests, on top of oracle/siglip_ref.py's stage helpers (which stay as they are).

Every function computes in its inputs' dtype, so float64 in gives a float64 reference; mode="autocast" rounds q and k to
bf16 before the fp32 softmax, as the encoder's bf16 path does."""
import torch

from oracle import siglip_ref as R


def _probs(q, k, H, ac, scale=None):
    """q [B,Nq,D], k [B,Nk,D] -> softmax(q kᵀ scale) per head [B,H,Nq,Nk]; the same arithmetic as oracle _mha's scores."""
    B, Nq, D = q.shape
    hd = D // H
    qh = R._rb(q, ac).view(B, Nq, H, hd).transpose(1, 2)
    kh = R._rb(k, ac).view(B, -1, H, hd).transpose(1, 2)
    s = (qh @ kh.transpose(-1, -2)) * (hd ** -0.5 if scale is None else scale)
    return torch.softmax(s, dim=-1)


@torch.no_grad()
def layer_attention_probs(sd: dict, c, i: int, h: torch.Tensor, mode: str = "fp32") -> torch.Tensor:
    """hidden_states[i] [B,N,D] -> encoder layer i's attention probabilities [B,H,N,N] (HF eager `attentions[i]`)."""
    ac = R._check_mode(mode)
    p = f"encoder.layers.{i}."
    y = R._layernorm(h, sd[p + "layer_norm1.weight"], sd[p + "layer_norm1.bias"], c.layer_norm_eps)
    q = R._linear(y, sd[p + "self_attn.q_proj.weight"], sd[p + "self_attn.q_proj.bias"], ac)
    k = R._linear(y, sd[p + "self_attn.k_proj.weight"], sd[p + "self_attn.k_proj.bias"], ac)
    return _probs(q, k, c.num_attention_heads, ac)


@torch.no_grad()
def map_probe_attention(sd: dict, c, last: torch.Tensor, mode: str = "fp32") -> torch.Tensor:
    """last_hidden_state [B,N,D] -> the MAP pooling probe's attention over the tokens [B,H,N]."""
    ac = R._check_mode(mode)
    B, D = last.shape[0], c.hidden_size
    wi, bi = sd["head.attention.in_proj_weight"], sd["head.attention.in_proj_bias"]
    probe = sd["head.probe"].reshape(1, 1, D).expand(B, 1, D)
    q = R._linear(probe, wi[:D], bi[:D], ac)
    k = R._linear(last, wi[D : 2 * D], bi[D : 2 * D], ac)
    return _probs(q, k, c.num_attention_heads, ac)[:, :, 0]


def attention_rollout(attn_mean: torch.Tensor, map_p: torch.Tensor, alpha: float = 0.5) -> torch.Tensor:
    """Attention rollout (Abnar & Zuidema 2020) seeded by the MAP probe: r = mean_h map_p [B,N], then for
    l = L-1 ... 0: r <- alpha·(r·attn_mean[l]) + (1 - alpha)·r, attn_mean [L,B,N,N] the head-mean probabilities.
    Every step is row-stochastic, so r sums to 1."""
    r = map_p.mean(dim=1)
    for l in range(attn_mean.shape[0] - 1, -1, -1):
        r = alpha * torch.einsum("bq,bqk->bk", r, attn_mean[l]) + (1.0 - alpha) * r
    return r

"""CPU tests of the attention maps (no GPU): the oracle's per-layer attention probabilities equal what the real
transformers SiglipVisionModel returns with output_attentions under eager attention, the oracle's rollout keeps its
invariants, and the new C-ABI entry points validate their arguments and fail loudly without a device."""
import ctypes as C

import pytest
import torch

from oracle import siglip_ref as R
from tests import attention_maps_ref as MR


@pytest.fixture(scope="module")
def lib():
    from dfd import _lib

    if not _lib.LIB_PATH.exists():
        import __graft_entry__ as g

        g.build()
    return _lib.load()


@pytest.mark.parametrize("name", ["tiny-hd64", "tiny-hd72", "small-hd72"])
def test_oracle_probs_equal_hf_eager_output_attentions(name):
    transformers = pytest.importorskip("transformers")
    c = R.CONFIGS[name]
    sd = R.init_state_dict(c, 0)
    hc = transformers.SiglipVisionConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                                         num_hidden_layers=c.num_hidden_layers, num_attention_heads=c.num_attention_heads,
                                         image_size=c.image_size, patch_size=c.patch_size)
    hc._attn_implementation = "eager"
    hf = transformers.SiglipVisionModel(hc).eval()
    hf.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
    x = R.preprocess_u8(R.synthetic_images(2, c.image_size, 3))
    with torch.no_grad():
        ref = hf(pixel_values=x, output_hidden_states=True, output_attentions=True)
    assert len(ref.attentions) == c.num_hidden_layers
    for i, a in enumerate(ref.attentions):
        p = MR.layer_attention_probs(sd, c, i, ref.hidden_states[i])
        assert p.shape == a.shape == (2, c.num_attention_heads, c.tokens, c.tokens)
        # 1e-6 absolute plus 1e-6 relative: both sides are fp32 with different reduction orders (worst measured:
        # 1.37e-6 at p = 0.88, small-hd72 layer 2)
        assert float(((p - a).abs() - 1e-6 * a).max()) <= 1e-6
    # the probe attention equals the weights of HF's MAP head (nn.MultiheadAttention, per head)
    mp = MR.map_probe_attention(sd, c, ref.last_hidden_state)
    assert mp.shape == (2, c.num_attention_heads, c.tokens)
    assert float((mp.sum(-1) - 1).abs().max()) <= 1e-6
    head = hf.vision_model.head
    with torch.no_grad():
        _, w = head.attention(head.probe.expand(2, -1, -1), ref.last_hidden_state, ref.last_hidden_state,
                              average_attn_weights=False)
    assert float((mp - w[:, :, 0]).abs().max()) <= 1e-6


def _random_stochastic(shape, g, dtype=torch.float64):
    a = torch.rand(shape, generator=g, dtype=dtype) ** 4
    return a / a.sum(-1, keepdim=True)


def test_oracle_rollout_invariants():
    g = torch.Generator().manual_seed(0)
    L, B, H, N = 4, 3, 5, 17
    A = _random_stochastic((L, B, N, N), g)
    mp = _random_stochastic((B, H, N), g)
    for alpha in (0.0, 0.3, 0.5, 1.0):
        r = MR.attention_rollout(A, mp, alpha)
        assert r.shape == (B, N)
        assert float((r.sum(-1) - 1).abs().max()) <= 1e-12
        assert bool((r >= 0).all())
    assert torch.equal(MR.attention_rollout(A, mp, 0.0), mp.mean(1))
    prod = A[L - 1]
    for l in range(L - 2, -1, -1):
        prod = prod @ A[l]
    want = torch.einsum("bq,bqk->bk", mp.mean(1), prod)
    assert float((MR.attention_rollout(A, mp, 1.0) - want).abs().max()) <= 1e-12
    # L = 0: the seed itself
    assert torch.equal(MR.attention_rollout(A[:0], mp, 0.5), mp.mean(1))


def test_abi_rejects_bad_arguments_without_a_device(lib):
    buf = (C.c_uint16 * (4 * 3 * 2 * 64 + 64))()
    p = (C.addressof(buf) + 15) // 16 * 16
    out = (C.c_float * 64)()
    o = C.addressof(out)
    # dfd_attention_probs(qkv, ldqkv, B, N, H, hd, scale, per_head, out, stream)
    assert lib.dfd_attention_probs(None, 384, 1, 4, 2, 64, 0.125, 1, o, None) == -1
    assert lib.dfd_attention_probs(p, 384, 1, 4, 2, 64, 0.125, 1, None, None) == -1
    assert lib.dfd_attention_probs(p, 432, 1, 4, 2, 72, 0.125, 1, o, None) in (-4, -5)  # valid: no device
    assert lib.dfd_attention_probs(p, 384, 1, 4, 2, 64, 0.125, 0, o, None) in (-4, -5)
    assert lib.dfd_attention_probs(p, 384, 1, 4, 2, 80, 0.125, 1, o, None) == -3        # head dim
    assert lib.dfd_attention_probs(p, 384, 1, 0, 2, 64, 0.125, 1, o, None) == -2        # N < 1
    assert lib.dfd_attention_probs(p, 384, 0, 4, 2, 64, 0.125, 1, o, None) == -2
    assert lib.dfd_attention_probs(p, 376, 1, 4, 2, 64, 0.125, 1, o, None) == -2        # ldqkv < 3·H·hd
    assert lib.dfd_attention_probs(p, 388, 1, 4, 2, 64, 0.125, 1, o, None) == -2        # ldqkv % 8
    assert lib.dfd_attention_probs(p, 384, 1, 4, 2, 64, 0.125, 2, o, None) == -1        # per_head
    assert lib.dfd_attention_probs(p, 384, 1, 4, 2, 64, 0.0, 1, o, None) == -1          # scale
    assert lib.dfd_attention_probs(p + 2, 384, 1, 4, 2, 64, 0.125, 1, o, None) == -1    # alignment
    # dfd_attention_rollout(attn_mean, map_p, L, B, N, H, alpha, G, S, relevance, heatmap, stream)
    assert lib.dfd_attention_rollout(None, o, 2, 1, 4, 2, 0.5, 2, 8, o, o, None) == -1
    assert lib.dfd_attention_rollout(o, None, 2, 1, 4, 2, 0.5, 2, 8, o, o, None) == -1
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 0.5, 2, 8, None, o, None) == -1
    assert lib.dfd_attention_rollout(o, o, 2, 1, 0, 2, 0.5, 2, 8, o, o, None) == -2     # N < 1
    assert lib.dfd_attention_rollout(o, o, -1, 1, 4, 2, 0.5, 2, 8, o, o, None) == -2    # L < 0
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 1.5, 2, 8, o, o, None) == -1     # alpha
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 0.5, 3, 8, o, o, None) == -2     # G·G != N
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 0.5, 2, 0, o, o, None) == -2     # S < 1
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 0.5, 2, 8, o, o, None) in (-4, -5)
    assert lib.dfd_attention_rollout(o, o, 2, 1, 4, 2, 0.5, 0, 0, o, None, None) in (-4, -5)  # no heatmap
    # dfd_engine_set_attention_tap(e, attn, per_head, map_p)
    assert lib.dfd_engine_set_attention_tap(None, o, 1, o) == -1
    assert lib.dfd_engine_set_attention_tap(None, None, 0, None) == -1
    assert lib.dfd_version() >= 102

"""GPU parity tests, kernel by kernel, through the C ABI (ctypes -> libdfd.so).

Floating-point kernels are compared against a plain fp32 torch restatement of the same op on the same
(bf16-rounded) inputs; tolerances are written next to each check.  Scoring kernels are compared against
oracle/scoring_ref.py and the reference-generated golden vectors (tests/golden/).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _bf(t):
    return t.to(torch.bfloat16)


def _gelu_tanh(x):
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


# ---------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------
GEMM_SHAPES = [
    # M, N, K                 what it is
    (256, 256, 128),          # smallest whole tiles
    (128, 128, 64),           # one tile, one k-block
    (1000, 768, 768),         # ragged M
    (392, 2304, 768),         # base qkv slice
    (300, 4304, 1152),        # so400m fc1: N not a multiple of any tile
    (300, 1152, 4304),        # so400m fc2: K not a multiple of 64 (TMA zero fill along K)
    (7, 1152, 640),           # tiny M (MAP head GEMMs, batch 7), padded patch K
    (1, 768, 768),            # single row
    (3000, 3456, 1152),       # so400m qkv, many tiles per CTA -> pipeline wrap-around and both accumulators
]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("tile_n", [0, 1128, 1192, 1256, 2128, 2192, 2256])  # auto, single-CTA, CTA-pair tiles
def test_gemm_plain(M, N, K, tile_n):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(M * 7 + N * 3 + K)
    a = _bf(torch.randn(M, K, generator=g)).to(DEV)
    w = _bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    out = ops.gemm_bf16(a, w, tile_n=tile_n)
    ref = a.float() @ w.float().t()
    torch.cuda.synchronize()
    # bf16 output rounding: 2^-9 relative; fp32 accumulation over K: negligible
    err = (out.float() - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 1e-3
    assert bool((err <= tol).all()), f"max err {err.max().item()} at {err.argmax().item()}"


@pytest.mark.parametrize("M,N,K", [(520, 768, 768), (300, 4304, 1152), (1458, 1152, 640)])
def test_gemm_epilogues(M, N, K):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(5)
    a = _bf(torch.randn(M, K, generator=g)).to(DEV)
    w = _bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    res = _bf(torch.randn(M, N, generator=g)).to(DEV)
    pos_rows = 729 if M % 729 == 0 else 13
    pos = torch.randn(pos_rows, N, generator=g).to(DEV)
    acc = a.float() @ w.float().t()

    def close(out, ref, what):
        err = (out.float() - ref).abs()
        tol = 2.0 ** -8 * ref.abs() + 2e-3
        assert bool((err <= tol).all()), f"{what}: max err {err.max().item()}"

    for tn in (1256, 2256, 2192):
        close(ops.gemm_bf16(a, w, bias=bias, residual=res, tile_n=tn), acc + bias + res.float(), f"bias+residual tile {tn}")
    close(ops.gemm_bf16(a, w, bias=bias), acc + bias, "bias")
    close(ops.gemm_bf16(a, w, bias=bias, act=1), _gelu_tanh(acc + bias), "bias+gelu_tanh")
    close(ops.gemm_bf16(a, w, bias=bias, residual=res), acc + bias + res.float(), "bias+residual")
    rows = torch.arange(M, device=DEV) % pos_rows
    close(ops.gemm_bf16(a, w, bias=bias, pos=pos), acc + bias + pos[rows], "bias+pos")
    # in-place residual (C aliases residual), as the engine uses it
    x = res.clone()
    ops.gemm_bf16(a, w, bias=bias, residual=x, out=x)
    close(x, acc + bias + res.float(), "in-place residual")
    # row statistics of the bf16 output: one (sum, sum of squares) partial per 64-column chunk, written (not accumulated)
    st = torch.full(((N + 63) // 64, M, 2), float("nan"), device=DEV)
    o = ops.gemm_bf16(a, w, bias=bias, stats_out=st)
    torch.cuda.synchronize()
    of = torch.nn.functional.pad(o.float(), (0, st.shape[0] * 64 - N)).view(M, -1, 64)
    assert torch.allclose(st[:, :, 0].t(), of.sum(2), rtol=1e-5, atol=1e-3)
    assert torch.allclose(st[:, :, 1].t(), (of * of).sum(2), rtol=1e-5, atol=1e-3)
    # bit-reproducible (no atomics): a second launch leaves identical statistics and output
    st2 = torch.empty_like(st)
    o2 = ops.gemm_bf16(a, w, bias=bias, stats_out=st2)
    assert torch.equal(st, st2) and torch.equal(o, o2)


@pytest.mark.parametrize("N,tile_n", [(1152, 2192), (1152, 1192), (320, 2256), (320, 1256), (1152, 2256), (192, 1128)])
def test_gemm_residual_many_tiles(N, tile_n):
    """Several tiles per CTA with a residual: the two epilogue groups drift apart, and with an odd number of
    64-column chunks per tile (tile 192, or an N tail of 1 or 3 chunks) they once shared residual slots."""
    from dfd import ops

    M, K = 148 * 128 * 5 + 77, 128
    g = torch.Generator(device="cpu").manual_seed(N + tile_n)
    a = _bf(torch.randn(M, K, generator=g)).to(DEV)
    w = _bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    res = _bf(torch.randn(M, N, generator=g)).to(DEV)
    ref = a.float() @ w.float().t() + res.float()
    for _ in range(3):
        out = ops.gemm_bf16(a, w, residual=res, tile_n=tile_n)
        torch.cuda.synchronize()
        err = (out.float() - ref).abs()
        bad = (err > 2.0 ** -8 * ref.abs() + 2e-3).nonzero()
        assert bad.numel() == 0, (f"{bad.shape[0]} wrong, max {err.max().item():.3f}, rows {bad[:, 0].min().item()}.."
                                  f"{bad[:, 0].max().item()} ({bad[:, 0].unique().numel()}), cols {bad[:, 1].min().item()}.."
                                  f"{bad[:, 1].max().item()}, row tiles {sorted(set((bad[:, 0] // 128).tolist()))[:10]}")


def test_gemm_ln_fold_whole_row_stats():
    """LayerNorm folded through the GEMM: LN(x)·(γ⊙W)ᵀ = rstd·(x·W'ᵀ − mean·colsum(W'))."""
    from dfd import ops

    M, D, N = 777, 1152, 384
    g = torch.Generator(device="cpu").manual_seed(9)
    x = _bf(torch.randn(M, D, generator=g) * 2.0 + 0.3).to(DEV)
    gamma = (1.0 + 0.1 * torch.randn(D, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(D, generator=g)).to(DEV)
    w = (torch.randn(N, D, generator=g) / math.sqrt(D)).to(DEV)
    b = torch.randn(N, generator=g).to(DEV)
    wf = _bf(w * gamma[None])
    colsum = wf.float().sum(1)
    bias2 = b + w @ beta
    xf = x.float()
    st = torch.stack([xf.sum(1), (xf * xf).sum(1)], -1).contiguous()   # [M, 2]: the ln_parts = 1 form
    out = ops.gemm_bf16(x, wf, bias=bias2, ln_rowstats=st, ln_colsum=colsum, ln_dim=D, ln_eps=1e-6)
    ref = torch.nn.functional.layer_norm(x.float(), (D,), gamma, beta, 1e-6) @ w.t() + b
    torch.cuda.synchronize()
    err = (out.float() - ref).abs().max().item()
    assert err < 0.06, err  # two bf16 roundings (W' and the output) on O(1) values


# The kernels bench.py times (so400m-384, B = 512 in chunks of <= 512 images => M > 9472 rows): CTA-pair 256-wide tiles with
# the compile-time epilogues EPI 1 (LN fold + bias: qkv), 2 (LN fold + bias + tanh-GELU: fc1), 3 (bias + residual + row
# statistics: out-projection / fc2), 4-6 (bias + residual / bias / bias + GELU with fuse_ln off), at the so400m shapes.
SO400M_GEMMS = [
    # name,   N,    K,    epi
    ("qkv", 3456, 1152, 1),
    ("fc1", 4304, 1152, 2),
    ("out", 1152, 1152, 3),
    ("fc2", 1152, 4304, 3),
    ("out_nostats", 1152, 1152, 4),
    ("qkv_noln", 3456, 1152, 5),
    ("fc1_noln", 4304, 1152, 6),
]


@pytest.mark.parametrize("name,N,K,epi", SO400M_GEMMS)
@pytest.mark.parametrize("M", [46656, 9600 + 77])  # 64 so400m images; just above the CTA-pair threshold with a ragged M tail
def test_gemm_specialised_epilogues_at_bench_shapes(name, N, K, epi, M):
    """fp32 torch reference on the same bf16 operands, row-sampled (every 97th row + the last 300) to keep the
    reference cheap; asserts that the <256, 2, *, EPI> instantiation is the kernel that ran."""
    from dfd import ops

    g = torch.Generator(device=DEV).manual_seed(N * 3 + K + epi)
    a = _bf(torch.randn(M, K, generator=g, device=DEV) * 1.5 + 0.25)
    w = _bf(torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K))
    bias = torch.randn(N, generator=g, device=DEV)
    rows = torch.cat([torch.arange(0, M, 97, device=DEV), torch.arange(M - 300, M, device=DEV)]).unique()
    af = a[rows].float()
    kw, ref = {}, None
    if epi in (1, 2):
        # LN folded through the GEMM; row statistics arrive as per-chunk partials, as the producer GEMM leaves them
        gamma = 1.0 + 0.1 * torch.randn(K, generator=g, device=DEV)
        beta = 0.1 * torch.randn(K, generator=g, device=DEV)
        wraw = w.float()
        w = _bf(wraw * gamma[None])
        colsum = w.float().sum(1)
        bias2 = bias + wraw @ beta
        parts = (K + 63) // 64
        ap = torch.nn.functional.pad(a.float(), (0, parts * 64 - K)).view(M, parts, 64)
        st = torch.stack([ap.sum(2), (ap * ap).sum(2)], -1).permute(1, 0, 2).contiguous()
        kw = dict(bias=bias2, ln_rowstats=st, ln_colsum=colsum, ln_dim=K, ln_eps=1e-6, act=1 if epi == 2 else 0)
        ref = torch.nn.functional.layer_norm(af, (K,), None, None, 1e-6) @ w.float().t() + bias2
        # (gamma is inside w already; LN without affine on the rows, then the folded weight: the same algebra in fp32)
        if epi == 2:
            ref = _gelu_tanh(ref)
    elif epi in (3, 4):
        res = _bf(torch.randn(M, N, generator=g, device=DEV))
        kw = dict(bias=bias, residual=res)
        if epi == 3:
            kw["stats_out"] = torch.full(((N + 63) // 64, M, 2), float("nan"), device=DEV)
        ref = af @ w.float().t() + bias + res[rows].float()
    else:
        kw = dict(bias=bias, act=1 if epi == 6 else 0)
        ref = af @ w.float().t() + bias
        if epi == 6:
            ref = _gelu_tanh(ref)
    out = ops.gemm_bf16(a, w, **kw)
    v = ops.gemm_last_variant()
    torch.cuda.synchronize()
    assert v == {"bn": 256, "cg": 2, "res": 1 if epi in (3, 4) else 0, "epi": epi}, v
    err = (out[rows].float() - ref).abs()
    # bf16 output (2^-9 relative) + tanh.approx GELU (5e-4 absolute) + the folded LN's two roundings
    tol = 2.0 ** -8 * ref.abs() + (6e-3 if epi in (1, 2) else 2e-3)
    assert bool((err <= tol).all()), f"{name}: max err {err.max().item()} (ref {ref.abs().max().item()})"
    if epi == 3:
        st = kw["stats_out"]
        of = torch.nn.functional.pad(out[rows].float(), (0, st.shape[0] * 64 - N)).view(rows.numel(), -1, 64)
        assert torch.allclose(st[:, rows, 0].t(), of.sum(2), rtol=1e-5, atol=1e-3)
        assert torch.allclose(st[:, rows, 1].t(), (of * of).sum(2), rtol=1e-5, atol=1e-3)
        assert torch.isfinite(st).all()   # every (chunk, row) slot was written
        # the consumer's view: LN statistics summed from the partials == statistics of the bf16 rows
        tot = st.sum(0)
        o_all = out.float()
        assert torch.allclose(tot[:, 0], o_all.sum(1), rtol=1e-5, atol=5e-2)
        assert torch.allclose(tot[:, 1], (o_all * o_all).sum(1), rtol=1e-4, atol=5e-2)


def test_gemm_ln_fold_outlier_channels():
    """The folded LayerNorm computes var = E[x²] − mean² in fp32 from per-chunk sums.  Real residual streams carry a few
    huge channels and rows with a common offset; this drives both (|mean| up to ~8 sigma of the bulk, channel outliers
    of 200 sigma) through the producer -> consumer pair at a CTA-pair shape and compares with fp32 LayerNorm."""
    from dfd import ops

    M, D, N = 12000, 1152, 512
    g = torch.Generator(device=DEV).manual_seed(77)
    x = torch.randn(M, D, generator=g, device=DEV)
    x[:, 7] += 200.0                                         # an always-on outlier channel
    x[:, 500] -= 120.0
    x += torch.linspace(-8, 8, M, device=DEV)[:, None]       # per-row common offset
    x[::5] *= 30.0                                           # high-norm tokens
    x = _bf(x)
    eye = _bf(torch.eye(D, device=DEV))
    st = torch.empty(((D + 63) // 64, M, 2), device=DEV)
    xo = ops.gemm_bf16(x, eye, bias=torch.zeros(D, device=DEV), residual=torch.zeros_like(x), stats_out=st, tile_n=2256)
    assert ops.gemm_last_variant()["epi"] == 3 and torch.equal(xo, x)
    gamma = 1.0 + 0.1 * torch.randn(D, generator=g, device=DEV)
    beta = 0.1 * torch.randn(D, generator=g, device=DEV)
    w = torch.randn(N, D, generator=g, device=DEV) / math.sqrt(D)
    b = torch.randn(N, generator=g, device=DEV)
    wf = _bf(w * gamma[None])
    out = ops.gemm_bf16(x, wf, bias=b + w @ beta, ln_rowstats=st, ln_colsum=wf.float().sum(1), ln_dim=D, ln_eps=1e-6,
                        tile_n=2256)
    assert ops.gemm_last_variant()["epi"] == 1
    ref = torch.nn.functional.layer_norm(x.float(), (D,), gamma, beta, 1e-6) @ w.t() + b
    torch.cuda.synchronize()
    err = (out.float() - ref).abs()
    # the reference LN output has channels of ~30 sigma here; tolerance = bf16 rounding of W' and of the output on that scale
    assert err.max().item() < 0.25 and err.mean().item() < 0.01, (err.max().item(), err.mean().item())


def test_gemm_bad_args():
    from dfd import _lib, ops

    a = torch.zeros(8, 12, dtype=torch.bfloat16, device=DEV)  # K % 8 != 0
    w = torch.zeros(8, 12, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(_lib.DfdError) as e:
        ops.gemm_bf16(a, w)
    assert e.value.code == -2


# ---------------------------------------------------------------------------------------------------
# LayerNorm / rowstats / patchify
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,D", [(1, 128), (37, 768), (1000, 1152), (513, 144), (64, 2048)])
def test_layernorm_bf16(M, D):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(D)
    x = _bf(torch.randn(M, D, generator=g) * 3 + 1).to(DEV)
    gamma = (1 + 0.2 * torch.randn(D, generator=g)).to(DEV)
    beta = (0.2 * torch.randn(D, generator=g)).to(DEV)
    y = ops.layernorm_bf16(x, gamma, beta, 1e-6)
    ref = torch.nn.functional.layer_norm(x.float(), (D,), gamma, beta, 1e-6)
    torch.cuda.synchronize()
    err = (y.float() - ref).abs()
    assert bool((err <= 2.0 ** -8 * ref.abs() + 1e-5).all()), err.max().item()


@pytest.mark.parametrize("S,P", [(224, 16), (384, 14), (60, 14)])
def test_patchify_u8(S, P):
    from dfd import ops
    from oracle import siglip_ref as R

    img = R.synthetic_images(3, S, seed=1)
    A = ops.patchify(img.to(DEV), S, P)
    x = R.preprocess_u8(img)
    G = S // P
    ref = x[:, :, : G * P, : G * P].reshape(3, 3, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(3 * G * G, 3 * P * P)
    torch.cuda.synchronize()
    K = 3 * P * P
    assert A.shape[1] % 64 == 0 and A.shape[1] >= K
    assert torch.equal(A[:, :K].cpu(), ref.to(torch.bfloat16)), "normalised patches must be bit-exact in bf16"
    assert float(A[:, K:].abs().max()) == 0.0 if A.shape[1] > K else True


@pytest.mark.parametrize("Hin,Win,skip", [(59, 57, 0), (56, 69, 1), (61, 60, 2)])
def test_patchify_u8_ragged_sides_and_unaligned_base(Hin, Win, skip):
    """Inputs anywhere on the 4x4 grid of a 60-pixel / patch-14 model (56..69-pixel sides, conv padding 'valid'), with the
    first image starting at an odd byte offset: the row-block kernel's 16-byte body + ragged ends must see every byte."""
    from dfd import ops

    S, P, G = 60, 14, 4
    g = torch.Generator().manual_seed(Hin * 100 + Win)
    flat = torch.randint(0, 256, (skip + 3 * Hin * Win * 3,), dtype=torch.uint8, generator=g).to(DEV)
    img = flat[skip:].view(3, Hin, Win, 3)
    assert img.data_ptr() % 16 == skip
    A = ops.patchify(img, S, P)
    x = (img.cpu().permute(0, 3, 1, 2).float() / 255.0 - 0.5) / 0.5
    ref = x[:, :, : G * P, : G * P].reshape(3, 3, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(3 * G * G, 3 * P * P)
    torch.cuda.synchronize()
    assert torch.equal(A[:, : 3 * P * P].cpu(), ref.to(torch.bfloat16))
    assert float(A[:, 3 * P * P:].abs().max()) == 0.0


@pytest.mark.parametrize("mode,name", [(1, "nearest"), (2, "bilinear")])
@pytest.mark.parametrize("Hin,S,P", [(32, 224, 16), (100, 60, 14), (300, 224, 16), (64, 60, 14)])  # 64: covers the 56-pixel patch grid but is not S: resampled, like the reference
def test_patchify_resize(mode, name, Hin, S, P):
    from dfd import ops
    from oracle import siglip_ref as R

    img = R.synthetic_images(2, Hin, seed=2)
    x = R.preprocess_u8(img)
    ref_img = R.resize_input(x, S, name)
    G = S // P
    ref = ref_img[:, :, : G * P, : G * P].reshape(2, 3, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(2 * G * G, -1)
    K = 3 * P * P
    for src in (img.to(DEV), x.to(DEV)):  # u8 NHWC and f32 NCHW inputs
        A = ops.patchify(src, S, P, resize_mode=mode)
        torch.cuda.synchronize()
        err = (A[:, :K].float().cpu() - ref).abs().max().item()
        assert err <= 2.0 ** -8 * 1.0 + 1e-6, err  # values in [-1,1], bf16 output


# ---------------------------------------------------------------------------------------------------
# attention
# ---------------------------------------------------------------------------------------------------
def _ref_attention(qkv, B, N, H, hd):
    D = H * hd
    q, k, v = (qkv.float()[:, i * D:(i + 1) * D].reshape(B, N, H, hd).transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * N, D)


@pytest.mark.parametrize("B,N,H,hd", [(2, 196, 12, 64), (1, 729, 16, 72), (3, 16, 2, 64), (2, 16, 2, 72),
                                      (2, 225, 4, 72), (1, 1024, 2, 72), (2, 64, 1, 64), (1, 129, 3, 64), (1, 1, 2, 72),
                                      (40, 576, 16, 64), (330, 100, 1, 72)])
@pytest.mark.parametrize("impl", [None, 5, 2])  # product dispatch; dual-query-tile; single-tile persistent
def test_attention(B, N, H, hd, impl):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(N + hd)
    qkv = _bf(torch.randn(B * N, 3 * H * hd, generator=g) * 1.5).to(DEV)
    out = ops.attention_bf16(qkv, B, N, H, hd, impl=impl)
    ref = _ref_attention(qkv, B, N, H, hd)
    torch.cuda.synchronize()
    err = (out.float() - ref).abs().max().item()
    # P is rounded to bf16 before PV (as in flash attention) and the output is bf16: ~2^-8 of |v| ~ 1.5·4
    assert err < 0.04, err
    assert torch.isfinite(out.float()).all()


def test_attention_large_logits_all_impls():
    """Rows whose max moves by far more than the lazy-rescale threshold between key tiles, and huge logits."""
    from dfd import ops

    B, N, H, hd = 2, 729, 2, 72
    g = torch.Generator(device="cpu").manual_seed(3)
    qkv = torch.randn(B * N, 3 * H * hd, generator=g) * 1.5
    qkv[:, :H * hd] *= 6.0                                   # sharp softmax
    qkv[N - 40:N, H * hd:2 * H * hd] *= 8.0                  # late keys dominate -> the running max jumps
    qkv = _bf(qkv).to(DEV)
    ref = _ref_attention(qkv, B, N, H, hd)
    for impl in (None, 5, 2):
        out = ops.attention_bf16(qkv, B, N, H, hd, impl=impl)
        torch.cuda.synchronize()
        assert torch.isfinite(out.float()).all()
        assert (out.float() - ref).abs().max().item() < 0.06, impl


@pytest.mark.parametrize("B,N,H,hd", [(3, 196, 12, 64), (2, 729, 16, 72), (5, 16, 2, 72), (1, 1024, 16, 72), (2, 1, 2, 72),
                                     (1, 3, 1, 64), (1, 4096, 2, 72),
                                     (13, 729, 16, 72), (64, 196, 12, 64)])   # so400m / base-224 heads at product batches
def test_map_attention(B, N, H, hd):
    """Against float64 on the same bf16 K | V (ldkv = 2·D, as the engine lays them out).  The outputs are weighted means of
    V, ~N^-1/2 in size, so the bound scales with the output: 2^-8·|ref| is the largest bf16 rounding of the result, and
    2^-12·max|v| leaves room for the fp32 accumulation.  Measured on a B200: worst |e| / bound 0.89, at N = 3 where rounding
    alone decides it; a P·V sum that drops one key exceeds the bound 10-300x."""
    from dfd import ops

    D = H * hd
    g = torch.Generator(device="cpu").manual_seed(N)
    kv = _bf(torch.randn(B * N, 2 * D, generator=g)).to(DEV)
    q = torch.randn(D, generator=g).to(DEV)
    k = kv.double()[:, :D].reshape(B, N, H, hd)
    v = kv.double()[:, D:].reshape(B, N, H, hd)
    for q_gain in (1.0, 2.0):   # 2.0: logits of std ~2, a sharp softmax
        qs = q * q_gain
        out = ops.map_attention_bf16(kv, qs, B, N, H, hd)
        s = torch.einsum("bnhd,hd->bhn", k, qs.double().reshape(H, hd)) / math.sqrt(hd)
        ref = torch.einsum("bhn,bnhd->bhd", torch.softmax(s, -1), v).reshape(B, D)
        err = (out.double() - ref).abs()
        bound = 2.0 ** -8 * ref.abs() + 2.0 ** -12 * v.abs().max()
        worst = float((err / bound).max())
        print(f"MAP B={B} N={N} H={H} hd={hd} q_gain={q_gain}: worst |e| / bound {worst:.3f}, "
              f"max |e| {float(err.max()):.2e}, rms |ref| {float(ref.square().mean().sqrt()):.3f}")
        assert worst <= 1.0, (q_gain, worst)


# ---------------------------------------------------------------------------------------------------
# classifier heads (golden vectors come from torch modules built exactly as the reference defines them)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [128, 1152])
def test_heads(D, golden_heads):
    from dfd import ops
    from dfd.pipeline import head_params_from_state
    from oracle import siglip_ref as R

    pooled = torch.from_numpy(golden_heads[f"pooled_{D}"])
    pb = pooled.to(torch.bfloat16).to(DEV)
    pr = pb.float().cpu()  # what the kernel actually sees
    protos = torch.from_numpy(golden_heads[f"protos_{D}"]).to(DEV)
    for kind, eps in (("A", 0.0), ("B", 1e-6)):
        sd = R.init_head(kind, D, 1)
        head = head_params_from_state(sd, D, DEV)
        assert head.kind == (1 if kind == "A" else 2)
        feats, z, pp = ops.head_fwd(head, pb, prototypes=protos, want_features=True)
        torch.cuda.synchronize()
        z_ref = R.classifier_head(sd, kind, pr, eps)
        assert torch.allclose(z.cpu(), z_ref, atol=2e-5, rtol=1e-5), (z.cpu() - z_ref).abs().max()
        # golden from the fp32 pooled: differs only by the bf16 rounding of the input (logit gate 1e-2)
        assert np.abs(z.cpu().numpy() - golden_heads[f"z{kind}_{D}"]).max() < 1e-2
        f_ref = R.l2_normalize(pr, eps)
        assert torch.allclose(feats.cpu(), f_ref, atol=1e-6)
        if kind == "A":
            p_ref = R.prototype_prob(f_ref, protos[0].cpu(), protos[1].cpu())
            assert torch.allclose(pp.cpu(), p_ref, atol=1e-5)
            assert np.abs(pp.cpu().numpy() - golden_heads[f"pproto_{D}"]).max() < 2e-3
    if D == 128:  # H-D (CiFake FastBinaryClassifier): LN -> one-token attention -> classifier, all four sizes
        for size in ("tiny", "small", "medium", "large"):
            sd = R.init_head_d(size, D, 4)
            z = ops.head_fwd(head_params_from_state(sd, D, DEV), pb)[1].cpu()
            assert torch.allclose(z, R.classifier_head_d(sd, pr), atol=2e-5, rtol=1e-5), size
            assert np.abs(z.numpy() - golden_heads[f"zD_{size}_{D}"]).max() < 1e-2
    # kind 0: normalise only
    head0 = ops.HeadParams(0, D, 0.0, DEV)
    feats, z, pp = ops.head_fwd(head0, pb, want_features=True)
    assert z is None and pp is None and torch.allclose(feats.cpu(), R.l2_normalize(pr, 0.0), atol=1e-6)


# ---------------------------------------------------------------------------------------------------
# frequency features
# ---------------------------------------------------------------------------------------------------
def _feat_close(v, ref, gray):
    from oracle import scoring_ref as S

    scale = np.maximum(np.abs(ref.astype(np.float64)), np.maximum(S.feature_scales(gray), 1e-12))
    return np.abs(v.astype(np.float64) - ref) / scale


def test_freq_features_golden(golden_scoring):
    """FreqMLP features within 1e-4 relative (BASELINE.json) of the reference's own extract_freq_vector."""
    from dfd import ops, scoring

    gray = golden_scoring["gray_u8"].astype(np.float32) / 255.0
    luts = scoring.build_freq_luts(DEV)
    x = torch.from_numpy(gray).to(DEV)
    raw = ops.freq_features(x, luts, eps=1e-8, zscore=False).cpu().numpy()
    zs = ops.freq_features(x, luts, eps=1e-8, zscore=True).cpu().numpy()
    for i in range(gray.shape[0]):
        rel = _feat_close(raw[i], golden_scoring["feats_raw"][i], gray[i])
        assert rel.max() < 1e-4, (i, int(rel.argmax()), rel.max(), raw[i], golden_scoring["feats_raw"][i])
        assert np.abs(zs[i] - golden_scoring["feats_zscore"][i]).max() < 1e-4


def test_freq_features_oracle_edge_cases():
    """Constant, impulse, single-frequency and random images against oracle/scoring_ref.py."""
    from dfd import ops, scoring
    from oracle import scoring_ref as S

    rng = np.random.default_rng(3)
    yy, xx = np.mgrid[0:256, 0:256]
    imgs = [np.zeros((256, 256), np.float32), np.full((256, 256), 0.5, np.float32),
            (rng.integers(0, 256, (256, 256)) / 255.0).astype(np.float32),
            (0.5 + 0.5 * np.cos(2 * np.pi * (8 * xx + 3 * yy) / 256)).astype(np.float32)]
    imp = np.zeros((256, 256), np.float32)
    imp[17, 200] = 1.0
    imgs.append(imp)
    x = torch.from_numpy(np.stack(imgs)).to(DEV)
    out = ops.freq_features(x, scoring.build_freq_luts(DEV)).cpu().numpy()
    assert np.isfinite(out).all()
    for i, im in enumerate(imgs):
        ref = S.extract_freq_vector(im)
        if i in (2,):  # generic image: the full gate
            assert _feat_close(out[i], ref, im).max() < 1e-4
        else:
            # degenerate spectra (exact zeros / a single line): phase of numerically-zero bins is arbitrary in any
            # FFT, so entropy (6), slope (4) and kurtosis of ~0 variance are excluded; the energy features must agree
            # (absolute floor 2e-5: an fp32 FFT's noise floor is ~1e-5 of the total spectral energy)
            for j in (0, 1, 2, 7, 8, 9, 10, 11, 12, 13, 14, 16, 19, 22):
                assert abs(out[i][j] - ref[j]) <= 1e-4 * abs(ref[j]) + 2e-5, (i, j, out[i][j], ref[j])


def test_freq_features_batch_consistency():
    """Large batch == per-image results (no cross-image leakage through scratch), bitwise for the energy
    features whose accumulation order is fixed."""
    from dfd import ops, scoring

    rng = np.random.default_rng(5)
    g = torch.from_numpy((rng.integers(0, 256, (67, 256, 256)) / 255.0).astype(np.float32)).to(DEV)
    luts = scoring.build_freq_luts(DEV)
    full = ops.freq_features(g, luts)
    for i in (0, 13, 66):
        one = ops.freq_features(g[i:i + 1].contiguous(), luts)
        assert torch.allclose(full[i], one[0], rtol=2e-5, atol=1e-7)
        assert torch.equal(full[i, 7:15], one[0, 7:15])


# ---------------------------------------------------------------------------------------------------
# score epilogue
# ---------------------------------------------------------------------------------------------------
def test_score_epilogue_g1_shipped(golden_scoring, shipped):
    """The shipped siglip/ artefacts end to end: FreqMLP G1 -> Linear(2,1) on probabilities -> temp -> CORAL."""
    from dfd import scoring
    from oracle import scoring_ref as S

    st = scoring.ScoringStack.from_dir(shipped["dir"], DEV)
    assert st.gen == 1
    feats = torch.from_numpy(golden_scoring["feats_zscore"]).to(DEV)
    z_sig = torch.linspace(-3, 3, feats.shape[0]).to(DEV)
    out = st(z_sig, feats=feats)
    torch.cuda.synchronize()
    zf = out["z_freq"].cpu().numpy()
    assert np.abs(zf - golden_scoring["zfreq_g1"]).max() < 2e-5
    z_ref = S.fusion_g1(shipped["fusion"], z_sig.cpu().numpy(), golden_scoring["zfreq_g1"])
    assert np.abs(out["z"].cpu().numpy() - z_ref).max() < 1e-5
    cl = S.coral_cut_logits(shipped["cuts"])
    d = S.detect_scores(z_ref, cl, shipped["temp"]["temperature"])
    for k in ("z_scaled", "p_raw", "p_coral", "entropy", "p_blend"):
        assert np.abs(out[k].cpu().numpy() - d[k]).max() < 1e-5, k
    assert np.abs(out["risk_probs"].cpu().numpy() - d["risk_probs"]).max() < 1e-6
    assert np.array_equal(out["risk_idx"].cpu().numpy(), d["risk_idx"])
    # survey known answers (SURVEY.md §8c(4)): z_sig in {-3,0,3} with z_freq=-6.5968 -> risk_idx 3
    zs3 = torch.tensor([-3.0, 0.0, 3.0], device=DEV)
    o3 = st(zs3, z_freq=torch.full((3,), -6.5968, device=DEV))
    assert np.allclose(o3["z_scaled"].cpu().numpy(), [0.21511, 0.54866, 0.88220], atol=2e-5)
    assert o3["risk_idx"].cpu().tolist() == [3, 3, 3]


def test_score_epilogue_g2(golden_scoring):
    from dfd import scoring
    from oracle import scoring_ref as S

    fs, hs = S.init_freq_mlp_g2(2), S.init_fusion_g2(3)
    cuts = [-1.0, -0.2, 0.3, 1.5]
    st = scoring.ScoringStack(DEV, fs, hs, cuts, 1.0)
    assert st.gen == 2
    feats = torch.from_numpy(golden_scoring["feats_raw"]).to(DEV)
    out = st(torch.zeros(feats.shape[0], device=DEV), feats=feats)
    assert np.abs(out["z_freq"].cpu().numpy() - golden_scoring["zfreq_g2"]).max() < 2e-5
    zs = torch.from_numpy(golden_scoring["fuse_zsig"]).to(DEV)
    zf = torch.from_numpy(golden_scoring["fuse_zfreq"]).to(DEV)
    out = st(zs, z_freq=zf)
    z = out["z"].cpu().numpy()
    assert np.abs(z - golden_scoring["fuse_g2_z"]).max() < 2e-5
    d = S.detect_scores(golden_scoring["fuse_g2_z"], np.array(cuts, np.float32), 1.0)
    tp = S.coral_transition_points(np.array(cuts, np.float32))
    near = np.abs(d["z_scaled"][:, None] - tp[None]).min(1) < 1e-2
    idx = out["risk_idx"].cpu().numpy()
    assert np.array_equal(idx[~near], d["risk_idx"][~near])
    assert len(set(idx.tolist())) >= 3  # these cuts reach several bins


def test_coral_sweep_against_reference(golden_scoring, shipped):
    """CORAL bin = argmax of sigmoid differences, identical to the reference's CoralCalibrator.predict on a
    z sweep, except within 1e-2 of an argmax transition point (SURVEY.md §A.6)."""
    from dfd import scoring
    from oracle import scoring_ref as S

    cal = scoring.CoralCalibrator(shipped["cuts"], device=DEV)
    assert np.allclose(cal.c.numpy(), golden_scoring["coral_cut_logits"], atol=1e-6)
    z = torch.from_numpy(golden_scoring["coral_z"]).to(DEV)
    idx, probs = cal.predict(z)
    idx, probs = idx.cpu().numpy(), probs.cpu().numpy()
    tp = S.coral_transition_points(golden_scoring["coral_cut_logits"])
    near = np.abs(golden_scoring["coral_z"][:, None] - tp[None]).min(1) < 1e-2
    assert np.array_equal(idx[~near], golden_scoring["coral_idx"][~near])
    assert np.abs(probs - golden_scoring["coral_probs"]).max() < 2e-6
    assert set(np.unique(idx)) == {0, 3, 4}
    i1, p1 = cal.predict(torch.tensor(0.5))
    assert i1 == 3 and p1.shape == (5,)


# ---------------------------------------------------------------------------------------------------
# fusion head training step
# ---------------------------------------------------------------------------------------------------
def test_fusion_fwd_bwd(golden_scoring):
    from dfd import ops
    from oracle import scoring_ref as S

    sd = S.init_fusion_g2(3)
    flat = torch.cat([sd[k].reshape(-1).float() for k in ops.FUSION_PARAM_ORDER]).to(DEV)
    zf = torch.from_numpy(golden_scoring["fuse_zfreq"]).to(DEV)
    zs = torch.from_numpy(golden_scoring["fuse_zsig"]).to(DEV)
    y = torch.from_numpy(golden_scoring["fuse_y"]).to(DEV)
    loss, grads, logits = ops.fusion_fwd_bwd(flat, zf, zs, y, want_logits=True)
    torch.cuda.synchronize()
    assert abs(loss.item() - float(golden_scoring["fuse_g2_loss"])) < 1e-5
    gr = golden_scoring["fuse_g2_grads"]
    assert np.abs(grads.cpu().numpy() - gr).max() < 1e-5 * max(1.0, np.abs(gr).max())
    assert np.abs(logits.cpu().numpy() - golden_scoring["fuse_g2_z"]).max() < 2e-5
    # linearity over shards: two half-batches with inv_global_batch = 1/B sum to the full-batch result
    l1, g1, _ = ops.fusion_fwd_bwd(flat, zf[:40].contiguous(), zs[:40].contiguous(), y[:40].contiguous(), 1.0 / 64)
    l2, g2, _ = ops.fusion_fwd_bwd(flat, zf[40:].contiguous(), zs[40:].contiguous(), y[40:].contiguous(), 1.0 / 64)
    assert torch.allclose(l1 + l2, loss, atol=1e-6) and torch.allclose(g1 + g2, grads, atol=1e-6)
    # large ragged batch vs float64 autograd oracle
    rng = np.random.default_rng(1)
    n = 10007
    zf2, zs2 = rng.normal(0, 3, n).astype(np.float32), rng.normal(0, 3, n).astype(np.float32)
    y2 = (rng.random(n) > 0.5).astype(np.float32)
    lo, go, _ = S.fusion_loss_and_grads(sd, zf2, zs2, y2)
    l3, g3, _ = ops.fusion_fwd_bwd(flat, torch.from_numpy(zf2).to(DEV), torch.from_numpy(zs2).to(DEV),
                                   torch.from_numpy(y2).to(DEV))
    assert abs(l3.item() - lo) < 1e-4 and np.abs(g3.cpu().numpy() - go).max() < 1e-4


# ---------------------------------------------------------------------------------------------------
# gray256 (Pillow luma + OpenCV CLAHE + Pillow bicubic resize): bit-exact
# ---------------------------------------------------------------------------------------------------
def test_gray256_matches_reference_golden(golden_gray):
    """dfd_gray256 against the outputs of the reference's own _pil_to_gray256[_clahe] on the seeded images."""
    from dfd import ops
    from oracle import gray_ref as G

    for i, (h, w, kind, seed) in enumerate(G.GOLDEN_CASES):
        rgb = torch.from_numpy(G.synthetic_rgb(h, w, kind, seed)).to(DEV)
        for j, clahe in enumerate((True, False)):
            got = ops.gray256_from_rgb(rgb[None].contiguous(), clahe)[0].cpu().numpy()
            want = golden_gray["gray_u8"][2 * i + j].astype(np.float32) / np.float32(255.0)
            assert np.array_equal(got, want), (h, w, kind, clahe, int((got != want).sum()))


@pytest.mark.parametrize("B,H,W", [(5, 384, 384), (3, 224, 224), (2, 100, 37), (1, 1, 1), (2, 600, 9),
                                   # the word-wide CLAHE / resample kernels: tile rows of 16 / 1 / 34 words, more than 8 taps per axis
                                   (2, 256, 512), (2, 40, 32), (1, 64, 1088), (2, 96, 160), (1, 768, 512)])
def test_gray256_batched_matches_oracle(B, H, W):
    from dfd import ops
    from oracle import gray_ref as G

    imgs = np.stack([G.synthetic_rgb(H, W, ("noise", "waves", "edges")[b % 3], 100 + b) for b in range(B)])
    for clahe in (True, False):
        got = ops.gray256_from_rgb(torch.from_numpy(imgs).to(DEV), clahe).cpu().numpy()
        for b in range(B):
            assert np.array_equal(got[b], G.gray256_from_rgb_u8(imgs[b], clahe)), (b, clahe)


def test_gray256_into_a_4_byte_aligned_output_and_scratch():
    """The word-wide kernels need 16-byte aligned output rows / 8-byte aligned scratch; pointers that are only 4-byte aligned take
    the generic kernels — same bits, no misaligned access."""
    from dfd import _lib, ops
    from oracle import gray_ref as G

    lib = _lib.load()
    B, H, W = 2, 64, 64
    imgs = np.stack([G.synthetic_rgb(H, W, "waves", 40 + b) for b in range(B)])
    want = np.stack([G.gray256_from_rgb_u8(im, True) for im in imgs])
    d = torch.from_numpy(imgs).to(DEV)
    out_buf = torch.zeros(B * 256 * 256 + 1, device=DEV)
    scr_buf = torch.zeros(lib.dfd_gray256_scratch_bytes(B, H, W) + 4, dtype=torch.uint8, device=DEV)
    got = ops.gray256_from_rgb(d, True, scratch=scr_buf[4:], out=out_buf[1:].view(B, 256, 256))
    assert got.data_ptr() % 16 == 4
    assert np.array_equal(got.cpu().numpy(), want)


def test_gray256_full_size_properties():
    """BASELINE batch (512 x 384 x 384): batch-permutation equivariance and range, no oracle at this size."""
    from dfd import ops

    g = torch.Generator(device=DEV).manual_seed(7)
    img = torch.randint(0, 256, (512, 384, 384, 3), dtype=torch.uint8, device=DEV, generator=g)
    a = ops.gray256_from_rgb(img, True)
    perm = torch.randperm(512, device=DEV, generator=g)
    b = ops.gray256_from_rgb(img[perm].contiguous(), True)
    assert torch.equal(a[perm], b)
    assert float(a.min()) >= 0.0 and float(a.max()) <= 1.0
    k = a.double() * 255.0
    assert float((k - k.round()).abs().max()) < 1e-4   # every value is k/255


@pytest.mark.parametrize("B,H,W,C", [(2, 384, 384, 3), (3, 100, 37, 3), (1, 257, 255, 3), (2, 64, 64, 1), (1, 8, 9, 3), (1, 1, 1, 3),
                                     (2, 480, 640, 3)])
def test_clahe_u8_per_channel_is_bit_exact(B, H, W, C):
    """dfd_clahe_u8 = `for c in range(3): arr[:, :, c] = clahe.apply(arr[:, :, c])` (train_fusion_head_only.py:60-65): against the
    numpy restatement of OpenCV's CLAHE (pinned to the library in tests/test_oracle_cpu.py) and, where installed, cv2 itself."""
    from dfd import ops
    from oracle import gray_ref as G

    imgs = np.stack([G.synthetic_rgb(H, W, ("noise", "waves", "edges")[b % 3], 300 + b) for b in range(B)])
    if C == 1:
        imgs = np.ascontiguousarray(imgs[..., 1:2])
    got = ops.clahe_u8(torch.from_numpy(imgs).to(DEV)).cpu().numpy()
    assert got.shape == imgs.shape and got.dtype == np.uint8
    for b in range(B):
        for c in range(C):
            want = G.clahe_u8(np.ascontiguousarray(imgs[b, :, :, c]))
            assert np.array_equal(got[b, :, :, c], want), (b, c, int((got[b, :, :, c] != want).sum()))
    try:
        import cv2
    except ImportError:
        return
    cl = cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8, 8))
    for b in range(B):
        for c in range(C):
            assert np.array_equal(got[b, :, :, c], cl.apply(np.ascontiguousarray(imgs[b, :, :, c])))


def test_device_preprocess_matches_reference_golden(golden_preprocess):
    """dfd_clahe_u8 + dfd_resize_u8 against the pixels of the reference's own `preprocess` object (train_fusion_head_only.py:60-74)
    and of its TTA transforms (inference_ai_human_images.py:195-215), generated in the build container by oracle/make_golden.py;
    the H-Flip view is the mirror of the Original one there, and here the patch kernel's DFD_FLIP_H read of the same pixels."""
    from dfd import ops, train_fusion
    from oracle import gray_ref as G

    g = golden_preprocess
    cases = [(97, 64, "noise", 5), (512, 384, "edges", 6), (300, 451, "waves", 4), (224, 224, "waves", 2)]
    S = int(g["tta_size"])
    for i, (h, w, kind, seed) in enumerate(cases):
        rgb = G.synthetic_rgb(h, w, kind, seed)
        d = torch.from_numpy(rgb).to(DEV)[None]
        got = ops.resize_u8(d, S, S, "bilinear")[0]
        assert np.array_equal(got.cpu().numpy(), g["tta_original_u8"][i]), ("tta", h, w)
        P = 16
        a_flip = ops.patchify(got[None].contiguous(), S, P, resize_mode=ops.FLIP_H)
        a_ref = ops.patchify(torch.from_numpy(np.ascontiguousarray(g["tta_original_u8"][i][:, ::-1])).to(DEV)[None], S, P)
        assert torch.equal(a_flip, a_ref)
        if i < len(g["train_u8"]):
            dev = train_fusion.preprocess_on_device(rgb, 384, torch.device(DEV))
            assert np.array_equal(dev.cpu().numpy(), g["train_u8"][i]), ("train", h, w)


def test_clahe_u8_rejects_in_place_and_bad_shapes():
    from dfd import _lib

    lib = _lib.load()
    x = torch.zeros(1, 16, 16, 3, dtype=torch.uint8, device=DEV)
    scr = torch.empty(lib.dfd_clahe_scratch_bytes(1, 3), dtype=torch.uint8, device=DEV)
    assert lib.dfd_clahe_u8(x.data_ptr(), 1, 16, 16, 3, scr.data_ptr(), x.data_ptr(), None) == -1    # DFD_ERR_BAD_ARG
    assert lib.dfd_clahe_u8(x.data_ptr(), 1, 16, 16, 2, scr.data_ptr(), scr.data_ptr(), None) == -2  # DFD_ERR_SHAPE
    assert lib.dfd_clahe_scratch_bytes(2, 3) == 2 * 3 * 64 * 256 and lib.dfd_clahe_scratch_bytes(0, 3) == 0


@pytest.mark.parametrize("B,H,W,OH,OW,C", [(3, 480, 640, 384, 384, 3), (4, 224, 224, 384, 384, 3), (2, 100, 37, 224, 224, 3),
                                           (1, 1080, 1920, 384, 384, 3), (2, 384, 384, 384, 384, 3), (3, 97, 211, 64, 48, 1)])
@pytest.mark.parametrize("filt", ["bilinear", "bicubic"])
def test_resize_u8_matches_pillow_oracle(B, H, W, OH, OW, C, filt):
    """dfd_resize_u8 = PIL Image.resize (torchvision transforms.Resize on PIL inputs), bit-exact."""
    from dfd import ops
    from oracle import gray_ref as G

    rng = np.random.default_rng(H + W + C)
    imgs = rng.integers(0, 256, (B, H, W, C), dtype=np.uint8)
    got = ops.resize_u8(torch.from_numpy(imgs).to(DEV), OH, OW, filt).cpu().numpy()
    for b in range(B):
        want = G.resize_u8(imgs[b] if C == 3 else imgs[b, ..., 0], OH, OW, filt)
        assert np.array_equal(got[b] if C == 3 else got[b, ..., 0], want), (b, filt)


def test_resize_then_patchify_equals_pil_preprocess():
    """a1 end to end on the device: PIL Resize((S,S)) + ToTensor + Normalize(.5,.5) == resize_u8 + patchify (bf16)."""
    from dfd import ops
    from oracle import gray_ref as G

    S, P = 224, 16
    rng = np.random.default_rng(5)
    imgs = rng.integers(0, 256, (2, 300, 451, 3), dtype=np.uint8)
    dev = ops.resize_u8(torch.from_numpy(imgs).to(DEV), S, S, "bilinear")
    A = ops.patchify(dev, S, P)
    ref_u8 = np.stack([G.resize_u8(im, S, S, "bilinear") for im in imgs])
    x = torch.from_numpy(ref_u8).permute(0, 3, 1, 2).float() / 255.0
    x = (x - 0.5) / 0.5
    g = S // P
    ref = x.reshape(2, 3, g, P, g, P).permute(0, 2, 4, 1, 3, 5).reshape(2 * g * g, 3 * P * P)
    torch.cuda.synchronize()
    assert torch.equal(A[:, :3 * P * P].float().cpu(), ref.to(torch.bfloat16).float())


# ---------------------------------------------------------------------------------------------------
# FreqMLP (G2) training step
# ---------------------------------------------------------------------------------------------------
def test_freqmlp_fwd_bwd(golden_freq_train):
    from dfd import ops
    from oracle import scoring_ref as S

    g = golden_freq_train
    sd = S.init_freq_mlp_g2(7)
    flat = torch.cat([torch.as_tensor(sd[k]).reshape(-1).float() for k in ops.FREQMLP_PARAM_ORDER]).to(DEV)
    mean, std = torch.as_tensor(sd["normer.mean"]).float().to(DEV), torch.as_tensor(sd["normer.std"]).float().to(DEV)
    feats, y = torch.from_numpy(g["feats"]).to(DEV), torch.from_numpy(g["y"]).to(DEV)
    loss, grads, logits = ops.freqmlp_fwd_bwd(flat, mean, std, feats, y, want_logits=True)
    torch.cuda.synchronize()
    # fp32 kernel vs the reference class's fp32 autograd: a few 1e-6 on O(1) values
    assert abs(loss.item() - float(g["loss"])) < 1e-5
    assert np.abs(grads.cpu().numpy() - g["grads"]).max() < 1e-5 * max(1.0, np.abs(g["grads"]).max())
    assert np.abs(logits.cpu().numpy() - g["logits"]).max() < 2e-5
    # eval-mode forward only
    _, _, lg = ops.freqmlp_fwd_bwd(flat, mean, std, feats, want_grads=False)
    assert torch.equal(lg, logits)
    # linearity over shards (what the data-parallel trainer relies on)
    l1, g1, _ = ops.freqmlp_fwd_bwd(flat, mean, std, feats[:20].contiguous(), y[:20].contiguous(), 1.0 / 37)
    l2, g2, _ = ops.freqmlp_fwd_bwd(flat, mean, std, feats[20:].contiguous(), y[20:].contiguous(), 1.0 / 37)
    assert torch.allclose(l1 + l2, loss, atol=1e-6) and torch.allclose(g1 + g2, grads, atol=2e-6)
    # large ragged batch vs the float64 oracle
    rng = np.random.default_rng(2)
    n = 5003
    f2 = (rng.normal(0.3, 0.8, (n, 24))).astype(np.float32)
    y2 = (rng.random(n) > 0.5).astype(np.float32)
    lo, go, _ = S.freq_mlp_g2_loss_and_grads(sd, f2, y2)
    l3, g3, _ = ops.freqmlp_fwd_bwd(flat, mean, std, torch.from_numpy(f2).to(DEV), torch.from_numpy(y2).to(DEV))
    assert abs(l3.item() - lo) < 1e-4 and np.abs(g3.cpu().numpy() - go).max() < 1e-4


def test_freqmlp_dropout_is_unbiased_and_seeded():
    from dfd import ops
    from oracle import scoring_ref as S

    sd = S.init_freq_mlp_g2(7)
    flat = torch.cat([torch.as_tensor(sd[k]).reshape(-1).float() for k in ops.FREQMLP_PARAM_ORDER]).to(DEV)
    mean, std = torch.as_tensor(sd["normer.mean"]).float().to(DEV), torch.as_tensor(sd["normer.std"]).float().to(DEV)
    g = torch.Generator(device="cpu").manual_seed(0)
    feats = (torch.randn(4096, 24, generator=g) * 0.8 + 0.3).to(DEV)
    y = (torch.rand(4096, generator=g) > 0.5).float().to(DEV)
    base = ops.freqmlp_fwd_bwd(flat, mean, std, feats, y)
    a = ops.freqmlp_fwd_bwd(flat, mean, std, feats, y, dropout_p=0.05, seed=1)
    b = ops.freqmlp_fwd_bwd(flat, mean, std, feats, y, dropout_p=0.05, seed=1)
    c = ops.freqmlp_fwd_bwd(flat, mean, std, feats, y, dropout_p=0.05, seed=2)
    assert torch.allclose(a[1], b[1], atol=1e-6)            # same seed, same masks (up to atomic ordering)
    assert not torch.allclose(a[1], c[1], atol=1e-6)        # different seed, different masks
    assert abs(a[0].item() - base[0].item()) < 0.2          # 5 % inverted dropout perturbs the loss only mildly


# ---------------------------------------------------------------------------------------------------
# SegFormer decoder pieces (SigLIP2_MTL)
# ---------------------------------------------------------------------------------------------------
def test_gemm_decoder_epilogues():
    """act 2 (erf GELU), act 3 (sigmoid) and the multiplicative residual (gate)."""
    from dfd import ops

    M, N, K = 700, 320, 256
    g = torch.Generator(device="cpu").manual_seed(21)
    a = _bf(torch.randn(M, K, generator=g)).to(DEV)
    w = _bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    x = _bf(torch.randn(M, N, generator=g)).to(DEV)
    acc = a.float() @ w.float().t() + bias

    def close(out, ref, what):
        err = (out.float() - ref).abs()
        assert bool((err <= 2.0 ** -8 * ref.abs() + 2e-3).all()), f"{what}: {err.max().item()}"

    close(ops.gemm_bf16(a, w, bias=bias, act=2), torch.nn.functional.gelu(acc), "gelu_erf")
    close(ops.gemm_bf16(a, w, bias=bias, act=3), torch.sigmoid(acc), "sigmoid")
    close(ops.gemm_bf16(a, w, bias=bias, act=3, residual=x, residual_op=1), torch.sigmoid(acc) * x.float(), "gate")
    # output into a column slice of a wider matrix (how the decoder concatenates its branches)
    wide = torch.zeros(M, 3 * N, dtype=torch.bfloat16, device=DEV)
    ops.gemm_bf16(a, w, bias=bias, act=2, out=wide[:, N:2 * N])
    close(wide[:, N:2 * N], torch.nn.functional.gelu(acc), "slice")
    assert float(wide[:, :N].abs().max()) == 0.0 and float(wide[:, 2 * N:].abs().max()) == 0.0


@pytest.mark.parametrize("B,H,W,E", [(2, 14, 14, 256), (3, 5, 7, 32), (1, 1, 1, 8), (2, 27, 27, 64)])
def test_dwconv3x3(B, H, W, E):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(H * W + E)
    x = _bf(torch.randn(B * H * W, E, generator=g))
    w = torch.randn(E, 1, 3, 3, generator=g) / 3
    b = torch.randn(E, generator=g)
    out = ops.dwconv3x3_bf16(x.to(DEV), w.reshape(E, 9).contiguous().to(DEV), b.to(DEV), B, H, W)
    ref = torch.nn.functional.conv2d(x.float().reshape(B, H, W, E).permute(0, 3, 1, 2), w, b, padding=1, groups=E)
    ref = ref.permute(0, 2, 3, 1).reshape(B * H * W, E)
    torch.cuda.synchronize()
    err = (out.float().cpu() - ref).abs()
    assert bool((err <= 2.0 ** -8 * ref.abs() + 1e-4).all()), err.max().item()


@pytest.mark.parametrize("B,H,S,E", [(2, 14, 224, 256), (3, 5, 70, 32), (1, 27, 384, 64), (2, 4, 4, 8)])
def test_seg_head_upsample(B, H, S, E):
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(H + S)
    x = _bf(torch.randn(B * H * H, E, generator=g))
    w = torch.randn(E, generator=g) / math.sqrt(E)
    out = ops.seg_head_upsample(x.to(DEV), w.to(DEV), 0.25, B, H, H, S).cpu()
    feat = x.float().reshape(B, H, H, E).permute(0, 3, 1, 2)
    up = torch.nn.functional.interpolate(feat, size=(S, S), mode="bilinear", align_corners=False)   # reference order:
    ref = torch.nn.functional.conv2d(up, w.reshape(1, E, 1, 1), torch.tensor([0.25]))              # upsample, then head
    assert (out - ref).abs().max() < 1e-4


def test_linear_small():
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(8)
    x = _bf(torch.randn(37, 1152, generator=g))
    w, b = torch.randn(3, 1152, generator=g) / 34, torch.randn(3, generator=g)
    out = ops.linear_small(x.to(DEV), w.to(DEV), b.to(DEV)).cpu()
    assert (out - (x.float() @ w.t() + b)).abs().max() < 1e-4


@pytest.mark.parametrize("M,N,K,tile_n", [(46656, 1152, 1152, 0), (20000, 1152, 4304, 0), (777, 768, 768, 0), (300, 264, 64, 1128),
                                          (1500, 1152, 256, 1192), (9000, 456, 128, 2128)])
def test_gemm_two_bf16_residual_stream(M, N, K, tile_n):
    """dfd_gemm_epilogue.residual_lo (EPI 7, every tile shape): v = A·Wᵀ + bias + hi + lo in fp32, C = hi' = bf16(v),
    lo' = bf16(v - hi') written back in place; hi' + lo' carries ~16 mantissa bits (2^-17 relative) where a bf16 stream keeps 8,
    and the row statistics are those of hi' (the operand the next LayerNorm-folded GEMM reads)."""
    from dfd import ops

    g = torch.Generator(device="cpu").manual_seed(M + N)
    a = _bf(torch.randn(M, K, generator=g)).to(DEV)
    w = _bf(torch.randn(N, K, generator=g) / K ** 0.5).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    x = (torch.randn(M, N, generator=g) * 3).to(DEV)                    # the "fp32" residual stream
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    ref = a.float() @ w.float().T + bias + hi.float() + lo.float()
    stats = torch.zeros(((N + 63) // 64, M, 2), dtype=torch.float32, device=DEV)
    out_hi, lo_t = hi.clone(), ops.lo_to_tiled(lo)
    assert torch.equal(ops.lo_from_tiled(lo_t, M, N), lo)
    ops.gemm_bf16(a, w, bias=bias, residual=out_hi, residual_lo=lo_t, stats_out=stats, out=out_hi, tile_n=tile_n)
    torch.cuda.synchronize()
    assert ops.gemm_last_variant()["epi"] == 7
    out_lo = ops.lo_from_tiled(lo_t, M, N)
    got = out_hi.float() + out_lo.float()
    scale = ref.abs().clamp_min(1.0)
    # fp32 accumulation order differs from torch's: allow 2e-5 relative for that; a one-tensor bf16 stream would sit at 2e-3
    assert float(((got - ref).abs() / scale).max()) < 6e-5
    assert float(((out_hi.float() - ref).abs() / scale).max()) < 4.1e-3          # hi' alone is the bf16 rounding of v
    st = stats.sum(0)
    assert torch.allclose(st[:, 0], out_hi.float().sum(1), rtol=1e-4, atol=1e-2)
    assert torch.allclose(st[:, 1], (out_hi.float() ** 2).sum(1), rtol=1e-4, atol=1e-2)
    # without statistics (the last layer's fc2)
    out_hi2, lo_t2 = hi.clone(), ops.lo_to_tiled(lo)
    ops.gemm_bf16(a, w, bias=bias, residual=out_hi2, residual_lo=lo_t2, out=out_hi2, tile_n=tile_n)
    torch.cuda.synchronize()
    assert torch.equal(out_hi2, out_hi) and torch.equal(lo_t2, lo_t)


def test_layernorm_bf16_with_lo():
    """layernorm over x = hi + lo (the post-LayerNorm of the precise engine mode) against fp32 torch."""
    from dfd import ops

    M, D = 1000, 1152
    g = torch.Generator(device="cpu").manual_seed(5)
    x = (torch.randn(M, D, generator=g) * 2 + 0.3).to(DEV)
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    gamma, beta = (1 + 0.1 * torch.randn(D, generator=g)).to(DEV), (0.1 * torch.randn(D, generator=g)).to(DEV)
    y = ops.layernorm_bf16(hi, gamma, beta, 1e-6, lo=ops.lo_to_tiled(lo))
    ref = torch.nn.functional.layer_norm(hi.float() + lo.float(), (D,), gamma, beta, 1e-6)
    torch.cuda.synchronize()
    assert float((y.float() - ref).abs().max()) < 2e-2       # bf16 output rounding of values up to ~4
    assert float((y.float() - ref).abs().mean()) <= float((ops.layernorm_bf16(hi, gamma, beta).float() - ref).abs().mean())


@pytest.mark.parametrize("clahe", [False, True])
def test_gray256_and_resize_on_rectangles_of_a_resident_image(clahe):
    """dfd_gray256 / dfd_resize_u8 on strided sources: a crop handed over as base pointer + strides (a torch view of the resident
    image, no copy) gives bit for bit what the dense kernels give on a contiguous copy of the crop — odd offsets, odd sizes,
    full-width slices at unaligned addresses, and a batch of same-size crops of a [B,H,W,3] stack."""
    from dfd import ops

    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (301, 413, 3), dtype=torch.uint8, generator=g).to(DEV)
    for (x0, y0, x1, y1) in [(0, 0, 413, 301), (7, 3, 260, 200), (101, 55, 413, 301), (0, 151, 413, 301), (33, 0, 34, 301),
                             (5, 9, 205, 10)]:
        view = img[y0:y1, x0:x1][None]
        dense = view.contiguous().clone()
        assert torch.equal(ops.gray256_from_rgb(view, clahe), ops.gray256_from_rgb(dense, clahe)), (x0, y0, x1, y1)
        for filt in ("bilinear", "bicubic"):
            assert torch.equal(ops.resize_u8(view, 60, 60, filt), ops.resize_u8(dense, 60, 60, filt)), (x0, y0, x1, y1, filt)
    stack = torch.randint(0, 256, (3, 120, 200, 3), dtype=torch.uint8, generator=g).to(DEV)
    view = stack[:, 11:97, 20:175]
    assert not view.is_contiguous()
    assert torch.equal(ops.gray256_from_rgb(view, clahe), ops.gray256_from_rgb(view.contiguous(), clahe))
    assert torch.equal(ops.resize_u8(view, 64, 48), ops.resize_u8(view.contiguous(), 64, 48))


# ---------------------------------------------------------------------------------------------------
# edge cases: empty / out-of-range inputs come back as status codes with a message, never as a launch
# ---------------------------------------------------------------------------------------------------
def test_c_abi_rejects_empty_and_out_of_range_shapes():
    """Every compute entry point validates its shape arguments before it touches the device: B = 0, M = 0, zero-sized images and
    unsupported head dims return DFD_ERR_SHAPE / DFD_ERR_UNSUPPORTED / DFD_ERR_BAD_ARG with text in dfd_last_error()."""
    from dfd import _lib

    lib = _lib.load()
    x = torch.zeros(4096, dtype=torch.uint8, device=DEV)
    p = x.data_ptr()
    launches = lib.dfd_launch_count()
    assert lib.dfd_gemm_bf16(p, 64, p, 64, p, 64, 0, 64, 64, None, None) == -2           # M = 0
    assert lib.dfd_gemm_bf16(p, 64, p, 64, p, 64, 8, 60, 64, None, None) == -2           # N not a multiple of 8
    assert lib.dfd_layernorm_bf16(p, 64, None, p, 64, p, p, 0, 64, 1e-6, None) == -2
    assert lib.dfd_attention_bf16(p, 192, p, 64, 0, 200, 1, 64, 0.125, None) == -2       # B = 0
    assert lib.dfd_attention_bf16(p, 3 * 80, p, 80, 1, 200, 1, 80, 0.1, None) == -3      # head dim 80: unsupported
    assert lib.dfd_freq_features(p, 0, p, 1e-8, 0, p, p, None) == -2
    assert lib.dfd_clahe_u8(p, 0, 8, 8, 3, p + 2048, p + 1024, None) == -2
    assert lib.dfd_gray256(p, 0, 0, 1, 0, 8, 1, p, p, p, 5, p, p, p, 5, p, p, None) == -2   # zero-height image
    assert lib.dfd_gray256_scratch_bytes(0, 8, 8) == 0 and lib.dfd_freq_scratch_bytes(0) == 0
    assert b":" in lib.dfd_last_error() or len(lib.dfd_last_error()) > 0
    assert lib.dfd_launch_count() == launches                                              # nothing was launched
    torch.cuda.synchronize()


def test_empty_batches_in_the_python_drivers():
    """The reference's loops over an empty loader / file list return empty results; so do the drop-in drivers."""
    from dfd import dropin, train_fusion

    class _M:
        resolution, device = 64, torch.device(DEV)

    assert train_fusion.extract_siglip_logits(_M(), []).shape == (0,)
    y, p, f = dropin.run_inference(None, [])
    assert y.shape == (0,) and p.shape == (0,) and f == []


def test_streaming_kernels_write_only_their_own_bytes():
    """Guard bands around every output and scratch buffer of the word-wide kernels (gray256, per-channel CLAHE, frequency
    features, patchify): sentinel bytes before and after each buffer survive the call (compute-sanitizer is not available on the
    pool; the results themselves are checked bit for bit by the tests above)."""
    from dfd import _lib, ops, scoring

    lib = _lib.load()
    G = 4096                                   # guard bytes on either side

    def guarded(nbytes, fill=0xA5):
        buf = torch.full((nbytes + 2 * G,), fill, dtype=torch.uint8, device=DEV)
        return buf, buf[G: G + nbytes]

    def intact(buf, nbytes, fill=0xA5):
        return bool((buf[:G] == fill).all()) and bool((buf[G + nbytes:] == fill).all())

    for (B, H, W) in [(3, 384, 384), (2, 224, 224), (2, 96, 160), (2, 100, 37)]:
        img = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=DEV)
        n_scr = lib.dfd_gray256_scratch_bytes(B, H, W)
        scr_buf, scr = guarded(n_scr)
        out_buf, out = guarded(B * 256 * 256 * 4)
        gray = ops.gray256_from_rgb(img, True, scratch=scr, out=out.view(torch.float32).view(B, 256, 256))
        torch.cuda.synchronize()
        assert intact(scr_buf, n_scr) and intact(out_buf, B * 256 * 256 * 4), ("gray256", B, H, W)
        # frequency features: scratch + [B,24] output
        n_f = lib.dfd_freq_scratch_bytes(B)
        f_buf, f_scr = guarded(n_f)
        luts = scoring.build_freq_luts(torch.device(DEV))
        feats = ops.freq_features(gray, luts, scratch=f_scr)
        torch.cuda.synchronize()
        assert intact(f_buf, n_f) and bool(torch.isfinite(feats).all()), ("freq", B)
        # per-channel CLAHE through the C ABI with guarded LUT scratch and destination
        n_l = lib.dfd_clahe_scratch_bytes(B, 3)
        l_buf, l_scr = guarded(n_l)
        d_buf, dst = guarded(B * H * W * 3)
        assert lib.dfd_clahe_u8(img.data_ptr(), B, H, W, 3, l_scr.data_ptr(), dst.data_ptr(), None) == 0
        torch.cuda.synchronize()
        assert intact(l_buf, n_l) and intact(d_buf, B * H * W * 3), ("clahe", B, H, W)
        assert torch.equal(dst.view(B, H, W, 3), ops.clahe_u8(img))
    for (S, P, B) in [(384, 14, 3), (224, 16, 2)]:
        img = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, device=DEV)
        Gd = S // P
        lda = (3 * P * P + 63) // 64 * 64
        n_a = B * Gd * Gd * lda * 2
        a_buf, a = guarded(n_a)
        assert lib.dfd_patchify(img.data_ptr(), 0, B, S, S, S, P, 0, a.data_ptr(), lda, None) == 0
        torch.cuda.synchronize()
        assert intact(a_buf, n_a), ("patchify", S, P)
        assert torch.equal(a.view(torch.bfloat16).view(B * Gd * Gd, lda), ops.patchify(img, S, P))

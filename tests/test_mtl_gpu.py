"""SigLIP2_MTL's tamper-mask decoder and class head against float64, kernel by kernel and stage by stage, on every GEMM tile
shape its epilogues run on.

The decoder is the only user of four GEMM epilogue options: erf-GELU (act 2), sigmoid (act 3), the multiplicative gate
(residual_op 1) and the store into a column slice of the concatenated [M, 4E] matrix.  Which kernel runs them depends on
M (gemm_tcgen05.cu pick_tile): at base-224 the decoder's GEMMs move to 256-row CTA pairs from B = 49 images up, where the
dispatch also holds compile-time specialised bias / bias + residual kernels that have no such options.  So

  * every decoder GEMM shape runs every one of these epilogues on every tile shape, at M on both sides of the CTA-pair
    threshold, and each call asserts that the generic kernel (EPI 0) of the expected tile ran;
  * the depthwise 3x3 convolution and the head + bilinear resize run at the decoder's grids and ratios;
  * the product configuration (base-224, seg_layers (2, 6, 10, -1), E = 256) is teacher-forced: every ops call of
    SegFormerStrongDecoder.forward is recorded and fed to float64 and bf16 emulation on its own inputs, with the gates of
    test_layers_gpu.py, and the whole chain is checked from the engine's hidden states to the seg logits.

Every reference is plain torch in float64 on the exact bf16 inputs the kernel received.  An error of the size of bf16
rounding cannot tell erf-GELU from tanh-GELU (they differ by at most 4.7e-4), so every erf-GELU output is also projected
onto d = gelu_tanh(z) - gelu_erf(z) of its float64 pre-activation z: the coefficient reads ~0 for erf and ~1 for tanh.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.test_layers_gpu import GEMM_VARIANTS, _by_images, _gate_ratios, no_tf32  # noqa: F401 (no_tf32: fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BASE = "siglip2-base-patch16-224"

# Worst values measured on a B200 (1000 W) over every case below, in brackets; each gate keeps >= 1.5x headroom.
GEMM_ABS = 1e-5       # |e| <= 2^-8 |ref| + GEMM_ABS for every decoder GEMM epilogue (4.4e-6)
GELU_PROJ = 0.15      # |<e, d> / <d, d>| of every erf-GELU output (0.070 at B = 1, where the emulation reads 0.071 by
                      # itself); tanh-GELU reads ~1
STAGE_ALPHA, STAGE_KAPPA, STAGE_BETA = 1.5, 1.5, 0.5   # the gates of test_layers_gpu.py for dwconv3x3 (border ring and
                                                       # interior each) and every teacher-forced decoder stage (1.000 /
                                                       # 1.000 / 0.001: the kernels round what the emulation rounds)
CHAIN_ALPHA, CHAIN_KAPPA, CHAIN_BETA = 1.6, 1.9, 7.0   # seg logits from the engine's hidden states (1.011 / 1.227 / 4.64)
SEG_TOL = 2e-6        # head + resize: |e| <= SEG_TOL * (the same op on |x|, |w|, |bias|) (8.0e-7, 14 -> 13)
CLS_TOL = 1e-7        # class head, likewise (2.3e-8)

# ---------------------------------------------------------------------------------------------------------------------
# GEMM epilogues
# ---------------------------------------------------------------------------------------------------------------------
TILES = [0, 1128, 1192, 1256, 2128, 2192, 2256]   # auto, then <bn, cg> forced: +1000 single CTA, +2000 CTA pair
# (name, K, N) of the decoder's GEMMs at base-224, E = 256: LinearProj, the 1x1 after the depthwise convolution,
# fuse_attn.0, fuse_attn.2 and fuse.0
DECODER_GEMMS = [("proj", 768, 256), ("pw", 256, 256), ("att0", 1024, 256), ("att2", 256, 1024), ("fuse", 1024, 256)]
# M = 196 B: 8 and 20 images run single-CTA tiles, 64 images and a 77-row tail run CTA pairs
GEMM_ROWS = [196 * 8, 196 * 20, 196 * 64 + 77]
# pick_tile's choice {(M, N): (bn, cg)} for the rows above
AUTO_TILE = {(1568, 256): (128, 1), (1568, 1024): (128, 1), (3920, 256): (128, 1), (3920, 1024): (256, 1),
             (12621, 256): (256, 2), (12621, 1024): (256, 2)}
# (act, multiplicative residual): erf-GELU (pw, att0), sigmoid, the gate sigmoid(.) * x (att2), and a plain product,
# which the C ABI accepts although the decoder does not issue it
EPILOGUES = [(2, False), (3, False), (3, True), (0, True)]
GUARD = 64   # guard columns on both sides of a sliced output / residual, guard rows below a sliced output


def _gelu_tanh(z):
    return 0.5 * z * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (z + 0.044715 * z ** 3)))


def _act(z, act):
    return {0: lambda t: t, 2: F.gelu, 3: torch.sigmoid}[act](z)


def _gemm_ref(a, w, bias, act, residual, residual_op, dt):
    """epi(a @ w^T + bias) in dtype dt, and the pre-activation."""
    z = a.to(dt) @ w.to(dt).t() + bias.to(dt)
    v = _act(z, act)
    if residual is not None:
        v = v * residual.to(dt) if residual_op else v + residual.to(dt)
    return v, z


def _gelu_projection(out, ref, z):
    """Coefficient of the error of an erf-GELU output along gelu_tanh(z) - gelu_erf(z)."""
    d = _gelu_tanh(z) - ref
    return float(((out.double() - ref) * d).sum() / (d * d).sum())


@pytest.mark.parametrize("tile_n", TILES)
def test_decoder_gemm_epilogues_every_tile(tile_n, no_tf32):
    from dfd import ops

    g = torch.Generator(device=DEV).manual_seed(tile_n + 1)
    worst_abs, worst_proj = 0.0, 0.0
    print(f"\nDECODER GEMMS tile_n={tile_n}: |e| - 2^-8 |ref| (worst over the epilogues), erf-GELU projections")
    for M in GEMM_ROWS:
        for name, K, N in DECODER_GEMMS:
            a = torch.randn(M, K, generator=g, device=DEV).to(torch.bfloat16)
            w = (torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).to(torch.bfloat16)
            bias = 0.5 * torch.randn(N, generator=g, device=DEV)
            r_wide = torch.randn(M, N + 2 * GUARD, generator=g, device=DEV).to(torch.bfloat16)
            r_dense = r_wide[:, GUARD:GUARD + N].contiguous()
            bn, cg = AUTO_TILE[(M, N)] if tile_n == 0 else (tile_n % 1000, tile_n // 1000)
            excess, projs = [], []
            for act, gate in EPILOGUES:
                for sliced in (False, True):
                    out = big = None
                    if sliced:   # a column slice of a wider matrix (ldc > N), with rows below it
                        big = torch.randn(M + 8, N + 2 * GUARD, generator=g, device=DEV).to(torch.bfloat16)
                        keep = big.clone()
                        out = big[:M, GUARD:GUARD + N]
                    res = (r_wide[:, GUARD:GUARD + N] if sliced else r_dense) if gate else None   # ldr > N when sliced
                    y = ops.gemm_bf16(a, w, bias=bias, act=act, residual=res, residual_op=int(gate), out=out,
                                      tile_n=tile_n)
                    v = ops.gemm_last_variant()
                    what = f"M={M} {name} act={act} gate={gate} sliced={sliced}"
                    ref, z = _gemm_ref(a, w, bias, act, res, 1, torch.float64)
                    excess.append(float((((y.double() - ref).abs() - 2.0 ** -8 * ref.abs())).max()))
                    assert excess[-1] <= GEMM_ABS, f"{what}: |e| exceeds 2^-8 |ref| by {excess[-1]:.3g}"
                    if act == 2:
                        projs.append(_gelu_projection(y, ref, z))
                        assert abs(projs[-1]) <= GELU_PROJ, f"{what}: erf-GELU projection {projs[-1]:+.3f}"
                    if sliced:
                        assert torch.equal(big[:, :GUARD], keep[:, :GUARD]), f"{what}: left guard columns written"
                        assert torch.equal(big[:, GUARD + N:], keep[:, GUARD + N:]), f"{what}: right guard columns written"
                        assert torch.equal(big[M:], keep[M:]), f"{what}: rows below M written"
                    assert (v["bn"], v["cg"], v["res"], v["epi"]) == (bn, cg, int(gate), 0), f"{what}: ran {v}"
            print(f"  M={M:5d} {name:4s} <{bn},{cg}>  excess {max(excess):+.2e}  gelu proj "
                  + " ".join(f"{p:+.4f}" for p in projs))
            worst_abs, worst_proj = max(worst_abs, max(excess)), max([worst_proj] + [abs(p) for p in projs])
    print(f"  worst excess {worst_abs:+.2e}, worst |gelu proj| {worst_proj:.4f}")


# ---------------------------------------------------------------------------------------------------------------------
# depthwise 3x3 convolution, head + bilinear resize
# ---------------------------------------------------------------------------------------------------------------------
def _dwconv_ref(x, w9, bias, B, H, W, dt):
    """Depthwise 3x3 convolution, zero padding 1, of token-major x [B·H·W, E] in dtype dt: a sum of nine shifted
    products (no convolution library, so nothing runs in TF32)."""
    E = x.shape[1]
    xp = F.pad(x.to(dt).view(B, H, W, E), (0, 0, 1, 1, 1, 1))
    out = bias.to(dt).expand(B, H, W, E).clone()
    for t in range(9):
        out += xp[:, t // 3:t // 3 + H, t % 3:t % 3 + W] * w9[:, t].to(dt)
    return out.view(B * H * W, E)


def _border(H, W):
    m = torch.zeros(H, W, dtype=torch.bool, device=DEV)
    m[0], m[-1], m[:, 0], m[:, -1] = True, True, True, True
    return m.flatten()


# grids 14 / 17 / 24 (224 / 280 / 384 px), 1 x 1 and 2 x 3; E = 256 (the decoder) and 64
DWCONV = [(64, 14, 14, 256), (1, 14, 14, 256), (43, 17, 17, 256), (21, 24, 24, 256), (64, 24, 24, 64), (7, 1, 1, 256),
          (9, 2, 3, 64), (5, 3, 2, 256)]


@pytest.mark.parametrize("B,H,W,E", DWCONV)
def test_dwconv3x3_border_and_interior(B, H, W, E):
    from dfd import ops

    g = torch.Generator(device=DEV).manual_seed(B * H * W + E)
    x = torch.randn(B * H * W, E, generator=g, device=DEV).to(torch.bfloat16)
    w9 = torch.randn(E, 9, generator=g, device=DEV) / 3
    bias = 0.1 * torch.randn(E, generator=g, device=DEV)
    out = ops.dwconv3x3_bf16(x, w9, bias, B, H, W)
    ref = _dwconv_ref(x, w9, bias, B, H, W, torch.float64)
    emu = _dwconv_ref(x, w9, bias, B, H, W, torch.float32)
    # the border ring (where padding enters) is a cell of its own, so that an error there is not diluted by the interior
    border = _border(H, W)
    for cell, m in (("border", border), ("interior", ~border)):
        if not bool(m.any()):
            continue
        pick = lambda t: t.view(B, H * W, E)[:, m]
        ratios = _gate_ratios(pick(out), pick(ref), pick(emu))
        print(f"\nDWCONV B={B} {H}x{W} E={E} {cell}: alpha / kappa / beta " + " / ".join(f"{r:.3f}" for r in ratios))
        assert ratios[0] <= STAGE_ALPHA and ratios[1] <= STAGE_KAPPA and ratios[2] <= STAGE_BETA, (cell, ratios)


def _seg_head_ref(f, w, bias, B, H, W, S, dt):
    """The reference's order (Siglip2sidafrozen.py:740-741): bilinear resize of every channel, then the 1x1 head."""
    E = f.shape[1]
    up = F.interpolate(f.to(dt).view(B, H, W, E).permute(0, 3, 1, 2), size=(S, S), mode="bilinear", align_corners=False)
    return (up * w.to(dt).view(1, E, 1, 1)).sum(1, keepdim=True) + bias


def _fp32_ratio(out, x, w, bias, f):
    """max |out - f(x, w, bias)| / f(|x|, |w|, |bias|), f in float64: the error in units of the op's own magnitude."""
    ref = f(x.double(), w.double(), bias)
    scale = f(x.double().abs(), w.double().abs(), abs(bias))
    return float(((out.double() - ref).abs() / scale).max())


# 14 -> 224, 17 -> 280, 24 -> 384 (the product sizes), 5 -> 70, 14 -> 14 and 14 -> 13 (a downsampling)
SEG_HEAD = [(2, 14, 224, 256), (2, 17, 280, 256), (2, 24, 384, 256), (3, 5, 70, 64), (4, 14, 14, 256), (3, 14, 13, 64)]


@pytest.mark.parametrize("B,H,S,E", SEG_HEAD)
def test_seg_head_upsample_vs_float64(B, H, S, E):
    from dfd import ops

    g = torch.Generator(device=DEV).manual_seed(H * S + E)
    x = torch.randn(B * H * H, E, generator=g, device=DEV).to(torch.bfloat16)
    w = torch.randn(E, generator=g, device=DEV) / math.sqrt(E)
    out = ops.seg_head_upsample(x, w, 0.25, B, H, H, S)
    r = _fp32_ratio(out, x, w, 0.25, lambda x_, w_, b_: _seg_head_ref(x_, w_, b_, B, H, H, S, torch.float64))
    print(f"\nSEG HEAD B={B} {H} -> {S} E={E}: |e| / scale {r:.2e}")
    assert r <= SEG_TOL


# ---------------------------------------------------------------------------------------------------------------------
# SigLIP2_MTL in the product configuration, teacher-forced
# ---------------------------------------------------------------------------------------------------------------------
class _Recorder:
    """Stands in for the ops module inside mtl: forwards every call and keeps the decoder's and the class head's inputs and
    outputs (copied, since the decoder writes into its concatenated matrix after the call), and for each GEMM the kernel
    instantiations it launched."""

    def __init__(self, ops):
        self._ops, self.calls = ops, []

    def __getattr__(self, name):
        return getattr(self._ops, name)

    def gemm_bf16(self, a, w, **kw):
        ops = self._ops
        res = kw.get("residual")
        res = None if res is None else res.clone()
        before = {k: ops.gemm_variant_launches(*k) for k in GEMM_VARIANTS}
        out = ops.gemm_bf16(a, w, **kw)
        ran = {k: n for k in GEMM_VARIANTS if (n := ops.gemm_variant_launches(*k) - before[k])}
        self.calls.append(("gemm", dict(a=a.clone(), w=w, bias=kw.get("bias"), act=kw.get("act", 0), residual=res,
                                        residual_op=kw.get("residual_op", 0), out=out.clone(), ran=ran)))
        return out

    def dwconv3x3_bf16(self, x, w9, bias, B, H, W):
        out = self._ops.dwconv3x3_bf16(x, w9, bias, B, H, W)
        self.calls.append(("dwconv", dict(x=x.clone(), w9=w9, bias=bias, B=B, H=H, W=W, out=out.clone())))
        return out

    def seg_head_upsample(self, x, w, bias, B, H, W, S):
        out = self._ops.seg_head_upsample(x, w, bias, B, H, W, S)
        self.calls.append(("head", dict(x=x.clone(), w=w, bias=bias, B=B, H=H, W=W, S=S, out=out.clone())))
        return out

    def linear_small(self, x, w, bias):
        out = self._ops.linear_small(x, w, bias)
        self.calls.append(("cls", dict(x=x.clone(), w=w, bias=bias, out=out.clone())))
        return out


STAGES = ["cls"] + [f"{s}{i}" for i in range(4) for s in ("proj", "dw", "pw")] + ["att0", "att2", "fuse", "head"]


def _chunks(calls):
    """The recorded calls of each forward chunk, {stage label: record}: the class head, then the decoder."""
    kinds = [k for k, _ in calls]
    one = [s if s in ("cls", "head") else ("dwconv" if s.startswith("dw") else "gemm") for s in STAGES]
    assert len(kinds) % len(one) == 0 and kinds == one * (len(kinds) // len(one)), kinds
    return [dict(zip(STAGES, (r for _, r in calls[i:i + len(one)]))) for i in range(0, len(calls), len(one))]


def _gemm_stage(r, dt):
    return _gemm_ref(r["a"], r["w"], r["bias"], r["act"], r["residual"], r["residual_op"], dt)


def _decoder_emu(st):
    """SegFormerStrongDecoder in bf16 emulation (fp32 math, outputs rounded to bf16 where the kernels store bf16), fed the
    recorded hidden states and the weights the kernels received."""
    rb = lambda t: t.to(torch.bfloat16).float()

    def gemm(r, a, residual=None):
        return rb(_gemm_ref(a, r["w"], r["bias"], r["act"], residual, r["residual_op"], torch.float32)[0])

    feats = []
    for i in range(4):
        d = st[f"dw{i}"]
        p = gemm(st[f"proj{i}"], st[f"proj{i}"]["a"])
        p = rb(_dwconv_ref(p, d["w9"], d["bias"], d["B"], d["H"], d["W"], torch.float32))
        feats.append(gemm(st[f"pw{i}"], p))
    cat = torch.cat(feats, 1)
    gated = gemm(st["att2"], gemm(st["att0"], cat), cat)
    h = st["head"]
    return _by_images(lambda f: _seg_head_ref(f, h["w"], h["bias"], f.shape[0] // (h["H"] * h["W"]), h["H"], h["W"],
                                              h["S"], torch.float32),
                      gemm(st["fuse"], gated), 8 * h["H"] * h["W"])


@pytest.fixture(scope="module")
def mtl_model():
    from dfd import mtl
    from oracle import decoder_ref as D
    from oracle import siglip_ref as R

    c = R.CONFIGS[BASE]
    sd = {"encoder.vision_model." + k: v for k, v in R.init_state_dict(c, 0).items()}
    sd.update(D.init_decoder_state(c.hidden_size, 4, 256, seed=1))
    model = mtl.SigLIP2_MTL(BASE, 0, max_batch=64).load_state_dict(sd)
    yield model, sd
    for eng in model._engines.values():
        eng.close()


# (image side, images, {(BN, CG, RES, EPI): launches} of the decoder's 12 GEMMs per forward).  Per chunk of B images:
# 4 LinearProj + fuse.0 (bias), 4 pointwise + fuse_attn.0 (bias + erf-GELU) on N = 256, fuse_attn.2 (sigmoid gate,
# residual) on N = 1024.  The bias-only GEMMs run the specialised EPI 5 on <256,2>, everything else the generic kernel.
MTL_ROWS = [
    pytest.param(224, 1, {(128, 1, 0, 0): 10, (128, 1, 1, 0): 1}, id="224px-B1"),
    pytest.param(224, 8, {(128, 1, 0, 0): 10, (128, 1, 1, 0): 1}, id="224px-B8"),
    pytest.param(224, 20, {(128, 1, 0, 0): 10, (256, 1, 1, 0): 1}, id="224px-B20"),
    # M = 12544: every decoder GEMM on CTA pairs
    pytest.param(224, 64, {(256, 2, 0, 5): 5, (256, 2, 0, 0): 5, (256, 2, 1, 0): 1}, id="224px-B64"),
    # max_batch 64: chunks of 64 and 6 images
    pytest.param(224, 70, {(256, 2, 0, 5): 5, (256, 2, 0, 0): 5, (256, 2, 1, 0): 1, (128, 1, 0, 0): 10,
                           (128, 1, 1, 0): 1}, id="224px-B70-chunked"),
    # the progressive-resize engines (grid 17 and 24, position table resampled)
    pytest.param(280, 8, {(128, 1, 0, 0): 10, (192, 1, 1, 0): 1}, id="280px-B8"),
    pytest.param(384, 8, {(128, 1, 0, 0): 10, (256, 1, 1, 0): 1}, id="384px-B8"),
]


def _compare(chunks, dsd, S, cls, seg):
    """Rows (stage, alpha, kappa, beta, erf-GELU projection of the kernel, of the emulation) for every bf16 stage of every
    chunk, (stage, |e| / scale) for the fp32 head + resize and the class head, and the chain's (alpha, kappa, beta) from
    the engine's hidden states to the seg logits `seg` (float64: the oracle's decoder)."""
    from oracle import decoder_ref as D

    rows, seg_ref, seg_emu = [], [], []
    for st in chunks:
        nb, grid = st["dw0"]["B"], st["dw0"]["H"]
        tok = lambda t: t.reshape(nb, grid * grid, -1)
        for k in STAGES[1:-1]:
            r = st[k]
            if k.startswith("dw"):
                ref = _dwconv_ref(r["x"], r["w9"], r["bias"], nb, grid, grid, torch.float64)
                emu = _dwconv_ref(r["x"], r["w9"], r["bias"], nb, grid, grid, torch.float32)
            else:
                ref, z = _gemm_stage(r, torch.float64)
                emu, _ = _gemm_stage(r, torch.float32)
            proj = (_gelu_projection(r["out"], ref, z), _gelu_projection(emu.to(torch.bfloat16), ref, z)) \
                if r.get("act") == 2 else (0.0, 0.0)
            rows.append((k, *_gate_ratios(tok(r["out"]), tok(ref), tok(emu)), *proj))
        h = st["head"]
        head = lambda x_, w_, b_: _by_images(
            lambda f: _seg_head_ref(f, w_, b_, f.shape[0] // (grid * grid), grid, grid, S, torch.float64), x_, 8 * grid * grid)
        rows.append(("head", _fp32_ratio(h["out"], h["x"], h["w"], h["bias"], head)))
        hidden = [tok(st[f"proj{i}"]["a"]).double() for i in range(4)]
        seg_ref.append(_by_images(lambda i: D.decoder_forward(dsd, [h_[i] for h_ in hidden], grid, S),
                                  torch.arange(nb, device=seg.device), 8))
        seg_emu.append(_decoder_emu(st))
    c = chunks[0]["cls"]
    pooled = torch.cat([st["cls"]["x"] for st in chunks])
    rows.append(("cls", _fp32_ratio(cls, pooled, c["w"], c["bias"], lambda x_, w_, b_: x_ @ w_.t() + b_.double())))
    px = lambda t: t.reshape(t.shape[0], S * S // 64, 64)
    chain = _gate_ratios(px(seg), px(torch.cat(seg_ref)), px(torch.cat(seg_emu)), stored=torch.float32)
    return rows, chain


@pytest.mark.parametrize("S,B,expect", MTL_ROWS)
def test_mtl_stages_vs_float64(S, B, expect, mtl_model, monkeypatch, no_tf32):
    from dfd import mtl, ops
    from oracle import siglip_ref as R

    model, sd = mtl_model
    rec = _Recorder(ops)
    monkeypatch.setattr(mtl, "ops", rec)
    cls, seg = model(R.synthetic_images(B, S, 7).to(DEV))
    monkeypatch.undo()
    torch.cuda.synchronize()
    chunks = _chunks(rec.calls)
    ran = {}
    for st in chunks:
        for k in STAGES:
            for v, n in st[k].get("ran", {}).items():
                ran[v] = ran.get(v, 0) + n
    dsd = {k: v.to(DEV, torch.float64) for k, v in sd.items() if k.startswith("decoder.")}
    rows, chain = _compare(chunks, dsd, S, cls, seg)

    print(f"\nMTL {S} px B={B}: stage alpha / kappa / beta, erf-GELU projection (engine, emulation); fp32 stages |e| / scale")
    for r in rows:
        if len(r) == 2:
            print(f"  {r[0]:5s} {r[1]:.2e}")
        else:
            print(f"  {r[0]:5s} {r[1]:6.3f} {r[2]:6.3f} {r[3]:7.3f}  {r[4]:+.4f} {r[5]:+.4f}")
    bf = [r for r in rows if len(r) == 6]
    print("  worst", " ".join(f"{max(r[j] for r in bf):6.3f}" for j in (1, 2, 3)),
          f" {max(abs(r[4]) for r in bf):.4f} {max(abs(r[5]) for r in bf):.4f}",
          f" head {max(r[1] for r in rows if r[0] == 'head'):.2e}")
    print(f"  chain: seg logits alpha / kappa / beta {chain[0]:.3f} / {chain[1]:.3f} / {chain[2]:.3f}")
    print(f"  decoder GEMM variants ran == expect: {ran == expect}")
    assert ran == expect, f"decoder GEMMs launched {ran}, expected {expect}"
    bad = [r for r in bf if r[1] > STAGE_ALPHA or r[2] > STAGE_KAPPA or r[3] > STAGE_BETA or abs(r[4]) > GELU_PROJ]
    assert not bad, f"stages over the gates (alpha {STAGE_ALPHA}, kappa {STAGE_KAPPA}, beta {STAGE_BETA}, projection " \
                    f"{GELU_PROJ}): {bad}"
    bad = [r for r in rows if len(r) == 2 and r[1] > (SEG_TOL if r[0] == "head" else CLS_TOL)]
    assert not bad, f"fp32 stages over the gates (head {SEG_TOL}, cls {CLS_TOL}): {bad}"
    assert chain[0] <= CHAIN_ALPHA and chain[1] <= CHAIN_KAPPA and chain[2] <= CHAIN_BETA, f"seg logits: {chain}"

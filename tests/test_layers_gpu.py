"""Stage-by-stage parity of the engine in the configurations bench.py runs, against a float64 reference.

The pooled-embedding gates of test_engine_gpu.py cannot see a defect smaller than the reference's own bf16 noise: one
attention head of one layer skipping a key tile moves that layer's output by ~0.16 and the pooled cosine by ~1e-5.  Here
every stage is teacher-forced: the engine's own bf16 input to a stage (the hidden-state tap) is fed to the oracle's code
for that stage in float64 and, for scale, in bf16 emulation (oracle mode "autocast", fp32, TF32 off).  With e the engine's
error and e_emu the emulation's error against float64, each stage must satisfy

  global       rms(e) <= ALPHA * rms(e_emu)
  per cell     rms(e) <= KAPPA * rms(e_emu) in every (image, 128-token row block, 64-column chunk), so a defect confined
               to one tile, chunk or image cannot hide in the global average
  elementwise  |e| <= 2^-7 |ref| + BETA * rms(e_emu)

These see a defect that is local or large.  A small systematic one spread over every element, such as a softmax scale off by
1 %, hides inside rounding noise of the same size; so every encoder layer also measures the logit scale its output implies:
the engine's error projected onto the float64 layer's response to a known change of the scale, which rounding noise (not
correlated with that response) leaves near zero.

The engine stores every stage's output in bf16, so the emulation's output is rounded to bf16 as well; otherwise the
residual stream, which the emulation keeps in fp32, would charge the engine for its storage format.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Worst values measured on a B200 over the four configurations below, every stage: alpha 1.41, kappa 1.49, beta 4.24, logit
# scale error 7.2e-4 (so400m; 1.4e-4 at base-224, 1.3e-4 for the bf16 emulation itself).  The gates keep >= 1.5x headroom.
ALPHA, KAPPA, BETA = 2.2, 2.4, 6.5
SCALE_STEP = 2.0 ** -7   # relative change of the logit scale whose response the layer error is projected onto
SCALE_TOL = 2e-3         # |relative logit scale error| an encoder layer may imply
ROW_BLOCK, COL_CHUNK = 128, 64

SO400M, BASE = "siglip2-so400m-patch14-384", "siglip2-base-patch16-224"


def _expected_gemms(L, fuse_ln, precise):
    """{(BN, CG, RES, EPI): launches} of the CTA-pair GEMM kernels in one forward of L layers.  The patch embedding (bias +
    pos, plus row statistics under fuse_ln) runs the generic kernel; the MAP head's K|V projection runs EPI 5."""
    if not fuse_ln:
        return {(256, 2, 0, 0): 1, (256, 2, 0, 5): L + 1, (256, 2, 0, 6): L, (256, 2, 1, 4): 2 * L}
    if precise:
        return {(256, 2, 0, 0): 1, (256, 2, 0, 1): L, (256, 2, 0, 2): L, (256, 2, 1, 7): 2 * L, (256, 2, 0, 5): 1}
    # the last layer's fc2 needs no row statistics: EPI 4 instead of 3
    return {(256, 2, 0, 0): 1, (256, 2, 0, 1): L, (256, 2, 0, 2): L, (256, 2, 1, 3): 2 * L - 1, (256, 2, 1, 4): 1,
            (256, 2, 0, 5): 1}


@pytest.fixture
def no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


def _cell_rms(e):
    """RMS of e [B, N, D] over each (image, ROW_BLOCK-token row block, COL_CHUNK-column chunk): [B, row blocks, chunks]."""
    B, N, D = e.shape
    assert D % COL_CHUNK == 0
    nb = -(-N // ROW_BLOCK)
    sq = torch.nn.functional.pad(e.square(), (0, 0, 0, nb * ROW_BLOCK - N))
    s = sq.view(B, nb, ROW_BLOCK, D // COL_CHUNK, COL_CHUNK).sum((2, 4))
    rows = torch.full((nb,), float(ROW_BLOCK), dtype=e.dtype, device=e.device)
    rows[-1] = N - (nb - 1) * ROW_BLOCK
    return (s / (rows[:, None] * COL_CHUNK)).sqrt()


def _gate_ratios(out, ref, emu):
    """(ALPHA, KAPPA, BETA) that the engine's output `out` needs: the smallest values with which it passes the gates."""
    if out.dim() == 2:   # pooled [B, D]: one row per image
        out, ref, emu = out[:, None], ref[:, None], emu[:, None]
    e = out.double() - ref
    e_emu = emu.to(torch.bfloat16).double() - ref
    rms_emu = e_emu.square().mean().sqrt()
    alpha = e.square().mean().sqrt() / rms_emu
    kappa = (_cell_rms(e) / _cell_rms(e_emu)).max()
    beta = ((e.abs() - 2.0 ** -7 * ref.abs()) / rms_emu).max()
    return float(alpha), float(kappa), float(beta)


def _scale_error(out, ref, ref_scaled):
    """Relative logit scale error implied by `out`: least-squares fit of out - ref onto the response ref_scaled - ref to a
    SCALE_STEP change of the scale."""
    e, g = out.double() - ref, ref_scaled - ref
    return float((e * g).sum() / (g * g).sum()) * SCALE_STEP


def _by_images(f, x, n):
    return torch.cat([f(x[i:i + n]) for i in range(0, x.shape[0], n)])


# so400m at B = 13 (M = 9477): the smallest batch on which every backbone GEMM, the D-wide out-projection / fc2 / patch
# embedding included, runs the 256-wide CTA-pair kernels that bench.py's batches run (at B = 16 those pick 192-wide
# tiles); its last CTA pair holds 5 rows.  base-224 at B = 64 (M = 12544).
@pytest.mark.parametrize("name,B,fuse_ln,precise", [(SO400M, 13, True, False), (SO400M, 13, True, True),
                                                    (BASE, 64, True, False), (BASE, 64, False, False)])
def test_every_stage_vs_float64(name, B, fuse_ln, precise, no_tf32):
    from dfd import engine, ops
    from oracle import siglip_ref as R

    c = R.CONFIGS[name]
    L = c.num_hidden_layers
    sd = R.init_state_dict(c, 0)
    eng = engine.SiglipEngine(engine.ARCHS[name], 0, max_batch=B, fuse_ln=fuse_ln,
                              precise_residual=precise).load_state_dict(sd)
    expect = _expected_gemms(L, fuse_ln, precise)
    before = {k: ops.gemm_variant_launches(*k) for k in expect}
    img = R.synthetic_images(B, c.image_size, 5).to(DEV)
    pooled, last, hidden = eng.forward_hidden(img)
    torch.cuda.synchronize()
    ran = {k: ops.gemm_variant_launches(*k) - before[k] for k in expect}
    eng.close()

    sd64 = {k: v.to(DEV, torch.float64) for k, v in sd.items()}
    sd32 = {k: v.to(DEV, torch.float32) for k, v in sd.items()}
    per = max(1, int(1e8 // (c.num_attention_heads * c.tokens ** 2 * 8)))   # images per chunk: float64 scores <= 100 MB
    rows = []

    def stage(label, f, x, out, scaled=None):
        ref = _by_images(lambda t: f(sd64, t.double(), "fp32"), x, per)
        emu = _by_images(lambda t: f(sd32, t.float(), "autocast"), x, per)
        ds = 0.0 if scaled is None else _scale_error(out, ref, _by_images(lambda t: scaled(sd64, t.double()), x, per))
        rows.append((label, *_gate_ratios(out, ref, emu), ds))

    stage("embed", lambda s, t, m: R.embed(s, c, t, m), R.preprocess_u8(img), hidden[0])
    for i in range(L):
        stage(f"layer {i}", lambda s, t, m: R.encoder_layer(s, c, i, t, m), hidden[i], hidden[i + 1],
              lambda s, t: R.encoder_layer(s, c, i, t, "fp32", c.head_dim ** -0.5 * (1 + SCALE_STEP)))
    stage("post-LN", lambda s, t, m: R.post_layernorm(s, c, t), hidden[L], last)
    stage("pooled", lambda s, t, m: R.map_head(s, c, t, m), last, pooled)

    print(f"\nSTAGES {name} B={B} fuse_ln={fuse_ln} precise={precise}: needed alpha / kappa / beta, logit scale error")
    for r in rows:
        print(f"  {r[0]:9s} {r[1]:6.3f} {r[2]:6.3f} {r[3]:7.3f} {r[4]:+.2e}")
    print("  worst    ", " ".join(f"{max(r[j] for r in rows):6.3f}" for j in (1, 2, 3)),
          f"{max(abs(r[4]) for r in rows):.2e}")
    assert ran == expect, f"CTA-pair GEMM kernels launched {ran}, expected {expect}"
    bad = [r for r in rows if r[1] > ALPHA or r[2] > KAPPA or r[3] > BETA or abs(r[4]) > SCALE_TOL]
    assert not bad, f"stages over the gates (alpha {ALPHA}, kappa {KAPPA}, beta {BETA}, scale {SCALE_TOL}): {bad}"

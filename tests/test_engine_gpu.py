"""End-to-end backbone parity on the GPU: dfd engine (C ABI) vs oracle/siglip_ref.py and the HF-generated
golden vectors, on seeded weights of the named architectures.

Gates (BASELINE.json): pooled embeddings cosine >= 0.999 against the reference path; additionally the
batch-mean-removed cosine and relative L2 are checked so a wrong-but-correlated result cannot pass.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _engine(name, max_batch, fuse_ln=False, precise=False):
    from dfd import engine
    from oracle import siglip_ref as R

    sd = R.init_state_dict(R.CONFIGS[name], 0)
    eng = engine.SiglipEngine(engine.ARCHS[name], 0, max_batch=max_batch, fuse_ln=fuse_ln,
                              precise_residual=precise).load_state_dict(sd)
    return eng, sd


@pytest.mark.parametrize("name,B", [("tiny-hd64", 3), ("tiny-hd72", 2), ("small-hd72", 2)])
def test_small_configs_vs_oracle_and_golden(name, B, golden_backbone):
    from oracle import siglip_ref as R

    c = R.CONFIGS[name]
    eng, sd = _engine(name, 4)
    img = R.synthetic_images(B, c.image_size, 0)
    pooled, last = eng(img.to(DEV), want_last_hidden=True)
    torch.cuda.synchronize()
    pooled, last = pooled.float().cpu(), last.float().cpu()
    ref = R.siglip_vision_forward(sd, c, R.preprocess_u8(img), "fp32")
    aut = R.siglip_vision_forward(sd, c, R.preprocess_u8(img), "autocast")
    gold = torch.from_numpy(golden_backbone[name + "/pooled"])
    for what, r in (("oracle fp32", ref["pooler_output"]), ("oracle autocast", aut["pooler_output"]), ("HF golden", gold)):
        rep = R.cosine_report(pooled, r)
        assert rep["cos_min"] >= 0.999, (what, rep)
        assert rep["cos_centered_min"] >= 0.995, (what, rep)
        assert rep["rel_l2"] <= 0.03, (what, rep)
    rep = R.cosine_report(last.reshape(-1, c.hidden_size), ref["last_hidden_state"].reshape(-1, c.hidden_size))
    assert rep["cos_min"] >= 0.998 and rep["rel_l2"] <= 0.03, rep
    gl = torch.from_numpy(golden_backbone[name + "/last_hidden_sub"])
    assert (last[:, ::7, ::5] - gl).abs().max() <= 0.03 * gl.abs().max() + 0.05


@pytest.mark.parametrize("name,B", [("tiny-hd64", 3), ("small-hd72", 2), ("siglip2-base-patch16-224", 2)])
def test_fused_layernorm_path(name, B, golden_backbone):
    """fuse_ln=1: LayerNorm1/2 folded into the qkv / fc1 GEMMs (gamma into the weights, (x-mean)*rstd through the
    epilogue, row statistics from the producing GEMM's epilogue).  Same gates as the unfused path; the two paths
    agree with each other to bf16 noise."""
    from oracle import siglip_ref as R

    c = R.CONFIGS[name]
    eng, sd = _engine(name, 4, fuse_ln=True)
    ref_eng, _ = _engine(name, 4, fuse_ln=False)
    img = R.synthetic_images(B, c.image_size, 0)
    pooled, last = eng(img.to(DEV), want_last_hidden=True)
    pooled0, _ = ref_eng(img.to(DEV))
    torch.cuda.synchronize()
    gold = torch.from_numpy(golden_backbone[name + "/pooled"])
    rep = R.cosine_report(pooled.float().cpu(), gold)
    assert rep["cos_min"] >= 0.999 and rep["cos_centered_min"] >= 0.995 and rep["rel_l2"] <= 0.04, rep
    rep2 = R.cosine_report(pooled.float().cpu(), pooled0.float().cpu())
    assert rep2["cos_min"] >= 0.9995 and rep2["rel_l2"] <= 0.03, rep2
    gl = torch.from_numpy(golden_backbone[name + "/last_hidden_sub"])
    assert (last.float().cpu()[:, ::7, ::5] - gl).abs().max() <= 0.04 * gl.abs().max() + 0.05
    # reloading weights into an engine whose tensors were folded in place must start from a full state dict
    eng.load_state_dict(sd)
    p2, _ = eng(img.to(DEV))
    assert R.cosine_report(p2.float().cpu(), pooled.float().cpu())["cos_min"] >= 0.9999


def test_f32_nchw_input_equals_u8_path():
    """The engine accepts already-normalised float tensors (what the reference's modules receive)."""
    from oracle import siglip_ref as R

    eng, _ = _engine("tiny-hd72", 4)
    img = R.synthetic_images(3, 60, 4)
    a, _ = eng(img.to(DEV))
    b, _ = eng(R.preprocess_u8(img).to(DEV))
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_chunking_and_determinism():
    from oracle import siglip_ref as R

    eng, _ = _engine("tiny-hd64", 4)
    img = R.synthetic_images(11, 64, 9).to(DEV)
    a, _ = eng(img)           # 3 chunks of <= 4
    b, _ = eng(img)
    c1, _ = eng(img[5:6])
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert torch.equal(a[5:6], c1), "an image's embedding must not depend on its batch neighbours"


@pytest.mark.parametrize("mode,name", [(1, "nearest"), (2, "bilinear")])
def test_in_model_resize(mode, name):
    """CiFake-style 32x32 inputs resampled inside the model (cifake_binary_classifier.py:716-717) and the
    default-nearest variant (train_fusion_head_only.py:103-104)."""
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd64"]
    eng, sd = _engine("tiny-hd64", 8)
    img = R.synthetic_images(5, 32, 3)
    pooled, _ = eng(img.to(DEV), resize_mode=mode)
    x = R.resize_input(R.preprocess_u8(img), c.image_size, name)
    ref = R.siglip_vision_forward(sd, c, x, "fp32")["pooler_output"]
    torch.cuda.synchronize()
    rep = R.cosine_report(pooled.float().cpu(), ref)
    assert rep["cos_min"] >= 0.999 and rep["rel_l2"] <= 0.03, rep


def test_base_224_vs_hf_golden(golden_backbone):
    """SigLIP-2 base-patch16-224 (BASELINE configs 1/2), B=2, against the HF fp32 forward."""
    from oracle import siglip_ref as R

    name = "siglip2-base-patch16-224"
    eng, sd = _engine(name, 8)
    assert abs(sum(float(v.double().sum()) for v in sd.values()) - float(golden_backbone[name + "/weight_checksum"])) < 1e-6
    img = R.synthetic_images(2, 224, 0)
    pooled, last = eng(img.to(DEV), want_last_hidden=True)
    torch.cuda.synchronize()
    gold = torch.from_numpy(golden_backbone[name + "/pooled"])
    rep = R.cosine_report(pooled.float().cpu(), gold)
    assert rep["cos_min"] >= 0.999 and rep["cos_centered_min"] >= 0.995 and rep["rel_l2"] <= 0.04, rep
    gl = torch.from_numpy(golden_backbone[name + "/last_hidden_sub"])
    assert (last.float().cpu()[:, ::7, ::5] - gl).abs().max() <= 0.04 * gl.abs().max() + 0.05


@pytest.mark.parametrize("fuse_ln", [False, True])  # True = the configuration bench.py measures
def test_base_224_logits(golden_backbone, fuse_ln):
    """BASELINE gate 'logits within 1e-2 absolute in bf16' at a named architecture: classifier heads H-A / H-B applied
    to the engine's pooled output vs the same heads (oracle, fp32) applied to the HF fp32 golden embedding."""
    from dfd import ops
    from dfd.pipeline import head_params_from_state
    from oracle import siglip_ref as R

    name = "siglip2-base-patch16-224"
    eng, _ = _engine(name, 8, fuse_ln=fuse_ln)
    pooled, _ = eng(R.synthetic_images(2, 224, 0).to(DEV))
    gold = torch.from_numpy(golden_backbone[name + "/pooled"])
    for kind, eps in (("A", 0.0), ("B", 1e-6)):
        hs = R.init_head(kind, 768, 1)
        z = ops.head_fwd(head_params_from_state(hs, 768, DEV), pooled)[1].cpu()
        z_ref = R.classifier_head(hs, kind, gold, eps)
        assert (z - z_ref).abs().max() < 1e-2, (kind, z, z_ref)


@pytest.mark.parametrize("fuse_ln", [False, True])
def test_so400m_384_vs_hf_golden(golden_backbone, fuse_ln):
    """SigLIP-2 so400m-patch14-384 (BASELINE config 3: 729 tokens, hd 72, I 4304), B=1, against HF fp32."""
    from oracle import siglip_ref as R

    name = "siglip2-so400m-patch14-384"
    eng, sd = _engine(name, 2, fuse_ln=fuse_ln)
    img = R.synthetic_images(1, 384, 0)
    pooled, last = eng(img.to(DEV), want_last_hidden=True)
    torch.cuda.synchronize()
    gold = torch.from_numpy(golden_backbone[name + "/pooled"])
    rep = R.cosine_report(pooled.float().cpu(), gold)
    assert rep["cos_min"] >= 0.999 and rep["rel_l2"] <= 0.04, rep
    gl = torch.from_numpy(golden_backbone[name + "/last_hidden_sub"])
    assert (last.float().cpu()[:, ::7, ::5] - gl).abs().max() <= 0.04 * gl.abs().max() + 0.05


def _hf_model(name, sd):
    import transformers

    from oracle import siglip_ref as R

    c = R.CONFIGS[name]
    hc = transformers.SiglipVisionConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                                         num_hidden_layers=c.num_hidden_layers,
                                         num_attention_heads=c.num_attention_heads, image_size=c.image_size,
                                         patch_size=c.patch_size)
    m = transformers.SiglipVisionModel(hc).eval()
    m.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
    return m.to(DEV)


GATE = {("siglip2-so400m-patch14-384", False): 1e-2, ("siglip2-so400m-patch14-384", True): 1e-2,
        ("siglip2-base-patch16-224", False): 1.25e-2, ("siglip2-base-patch16-224", True): 1e-2}
BENCH_KERNELS = ((256, 2, 0, 1), (256, 2, 0, 2), (256, 2, 1, 3))   # qkv (LN fold), fc1 (LN fold + GELU), out / fc2 (+stats)
PRECISE_KERNELS = ((256, 2, 0, 1), (256, 2, 0, 2), (256, 2, 1, 7))  # the same on the two-bf16 residual stream


@pytest.mark.parametrize("name,B,S,precise", [("siglip2-so400m-patch14-384", 64, 384, False),
                                              ("siglip2-so400m-patch14-384", 64, 384, True),
                                              ("siglip2-base-patch16-224", 64, 224, False),
                                              ("siglip2-base-patch16-224", 64, 224, True)])
def test_benched_configuration_vs_hf_on_gpu(name, B, S, precise):
    """The configuration bench.py times — fuse_ln on, M = B·N > 9472 token rows, i.e. the CTA-pair GEMM kernels with the
    compile-time LN-fold / GELU / residual+statistics epilogues and the dual-query-tile attention kernel — against the
    reference path itself: transformers.SiglipVisionModel on this GPU, in fp32 (TF32 off) and under bf16 autocast
    (inference_ai_human_images.py:267,279 runs the backbone under autocast).  Gates of BASELINE.json: pooled cosine
    >= 0.999 (plus the batch-mean-removed cosine >= 0.995), H-A / H-B logits within 1e-2."""
    pytest.importorskip("transformers")
    from dfd import ops
    from dfd.pipeline import head_params_from_state
    from oracle import siglip_ref as R

    eng, sd = _engine(name, B, fuse_ln=True, precise=precise)
    kernels = PRECISE_KERNELS if precise else BENCH_KERNELS
    before = [ops.gemm_variant_launches(*k) for k in kernels]
    img = R.synthetic_images(B, S, 11)
    pooled, _ = eng(img.to(DEV))
    torch.cuda.synchronize()
    L = R.CONFIGS[name].num_hidden_layers
    ran = [ops.gemm_variant_launches(*k) - b for k, b in zip(kernels, before)]
    # (the last layer's fc2 needs no row statistics: EPI 4 in the default mode, EPI 7 without stats_out in the precise one)
    expect = [L, L, 2 * L] if precise else [L, L, 2 * L - 1]
    assert ran == expect, f"specialised kernels launched {ran}, expected {expect}"
    pooled2, _ = eng(img.to(DEV))
    assert torch.equal(pooled, pooled2), "the fused-LayerNorm path must be bit-reproducible (no atomics)"

    m = _hf_model(name, sd)
    x = R.preprocess_u8(img).to(DEV)
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            hf32 = torch.cat([m(pixel_values=x[i:i + 8]).pooler_output for i in range(0, B, 8)]).float().cpu()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                hf16 = torch.cat([m(pixel_values=x[i:i + 8]).pooler_output for i in range(0, B, 8)]).float().cpu()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    del m
    ours = pooled.float().cpu()
    for what, ref in (("HF fp32", hf32), ("HF bf16 autocast", hf16)):
        rep = R.cosine_report(ours, ref)
        assert rep["cos_min"] >= 0.999 and rep["cos_centered_min"] >= 0.995 and rep["rel_l2"] <= 0.04, (what, rep)
    noise = R.cosine_report(hf16, hf32)   # the reference's own bf16 noise, for scale
    D = R.CONFIGS[name].hidden_size
    worst = {}
    for kind, eps in (("A", 0.0), ("B", 1e-6)):
        hs = R.init_head(kind, D, 1)
        z = ops.head_fwd(head_params_from_state(hs, D, DEV), pooled)[1].cpu()
        z32, z16 = R.classifier_head(hs, kind, hf32, eps), R.classifier_head(hs, kind, hf16, eps)
        worst[kind] = (float((z - z32).abs().max()), float((z - z16).abs().max()), float((z16 - z32).abs().max()))
    print(f"PARITY {name} B={B} precise={precise}: logit |d| vs fp32 / vs autocast / autocast vs fp32 = {worst}; rel_l2 ours "
          f"{R.cosine_report(ours, hf32)['rel_l2']:.4f} HF-autocast {noise['rel_l2']:.4f}")
    for kind in worst:
        # gate: within 1e-2 of the fp32 reference logits (the reference's own autocast path sits worst[kind][2] away from them)
        assert worst[kind][0] <= GATE[(name, precise)], (kind, worst, noise)
        assert worst[kind][1] <= 1.5e-2, (kind, worst, noise)   # two independent bf16 paths: noise adds
    eng.close()


def test_detect_records_at_batch_512_equal_small_batch_records():
    """BASELINE config 3 at full size (so400m-384, 512 images per step, fuse_ln on), through the whole pipeline: the score
    records of 64 sampled images inside the 512-image step are bit-identical to a 64-image step of the same images
    (M = 46 656 token rows: the same CTA-pair kernels as the 512-image step, other tile schedule; an image's result
    does not depend on its batch neighbours or on the schedule), and 16 of them agree with the unfused small-batch path (generic kernels, LayerNorm as its own kernel) to bf16 noise with CORAL
    indices identical outside the transition band."""
    from dfd import pipeline, scoring, weights
    from dfd.engine import ARCHS
    from oracle import siglip_ref as R

    name = "siglip2-so400m-patch14-384"
    arch = ARCHS[name]
    bsd = weights.random_vision_state_dict(arch, seed=0, device=torch.device(DEV))
    head = weights.random_classifier_head("B", arch.hidden_size, 1)

    def make(fuse, mb):
        st = scoring.ScoringStack(torch.device(DEV), weights.random_freq_mlp_g2(2), weights.random_fusion_g2(3),
                                  [-1.0, -0.2, 0.3, 1.5], 1.0)
        return pipeline.DetectionPipeline(arch, bsd, head, st, device=0, max_batch=mb, fuse_ln=fuse)

    img = R.synthetic_images(512, 384, 5).to(DEV)
    big = make(True, 512)
    rec512 = big.pack(big.detect_device(img, None, clahe=True)).cpu()
    idx64 = torch.arange(3, 512, 8)[:64]
    rec64 = big.pack(big.detect_device(img[idx64.to(DEV)].contiguous(), None, clahe=True)).cpu()
    assert torch.isfinite(rec512).all()
    f = pipeline.PACKED_FIELDS
    # backbone + head: bit-identical.  The frequency branch is not batch-invariant to the last bit (freq_cols_kernel splits
    # an image's column groups over a batch-dependent number of CTAs, so its fp32 partial sums add in another order:
    # ~1e-6), and everything downstream of z_freq inherits that.
    assert torch.equal(rec512[idx64][:, f.index("z_sig")], rec64[:, f.index("z_sig")])
    assert torch.allclose(rec512[idx64], rec64, rtol=0, atol=2e-5), (rec512[idx64] - rec64).abs().max()
    idx = idx64[:16]
    sub = img[idx.to(DEV)].contiguous()
    rec16 = rec64[:16]
    del big
    torch.cuda.empty_cache()
    small = make(False, 4)
    rec_ref = small.pack(small.detect_device(sub, None, clahe=True)).cpu()
    dz = (rec16[:, f.index("z_sig")] - rec_ref[:, f.index("z_sig")]).abs().max()
    assert dz <= 1e-2, dz
    assert torch.allclose(rec16[:, f.index("z_freq")], rec_ref[:, f.index("z_freq")], rtol=0, atol=2e-5)   # fp32 feature path
    # CORAL: identical unless z_scaled sits within the logit tolerance of an argmax transition point
    zs, ia, ib = rec_ref[:, f.index("z_scaled")], rec16[:, f.index("risk_idx")], rec_ref[:, f.index("risk_idx")]
    import numpy as np

    from oracle import scoring_ref as S

    trans = S.coral_transition_points(np.array([-1.0, -0.2, 0.3, 1.5], np.float32))
    for i in range(16):
        if ia[i] != ib[i]:
            assert min(abs(float(zs[i]) - float(t)) for t in trans) <= 1e-2, (i, zs[i], ia[i], ib[i])


def test_full_size_properties_batch_256():
    """At BASELINE size (base-224, batch 256) the oracle is too slow; use size-independent properties:
    permutation equivariance over the batch and equality with the small-batch result."""
    from oracle import siglip_ref as R

    eng, _ = _engine("siglip2-base-patch16-224", 256)
    img = R.synthetic_images(256, 224, 1).to(DEV)
    a, _ = eng(img)
    perm = torch.randperm(256, generator=torch.Generator().manual_seed(0)).to(DEV)
    b, _ = eng(img[perm].contiguous())
    s, _ = eng(img[:2].contiguous())
    torch.cuda.synchronize()
    assert torch.isfinite(a.float()).all()
    assert torch.equal(a[perm], b)
    assert torch.equal(a[:2], s)


def test_hf_bf16_autocast_on_gpu(golden_backbone):
    """The literal 'reference PyTorch/HF path in bf16' of BASELINE.json, run on this GPU (transformers is part of
    the image, not of /root/reference): pooled cosine >= 0.999."""
    transformers = pytest.importorskip("transformers")
    from oracle import siglip_ref as R

    name = "siglip2-base-patch16-224"
    c = R.CONFIGS[name]
    eng, sd = _engine(name, 8)
    hc = transformers.SiglipVisionConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                                         num_hidden_layers=c.num_hidden_layers,
                                         num_attention_heads=c.num_attention_heads, image_size=c.image_size,
                                         patch_size=c.patch_size)
    m = transformers.SiglipVisionModel(hc).eval()
    m.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
    m = m.to(DEV)
    img = R.synthetic_images(8, 224, 2)
    x = R.preprocess_u8(img).to(DEV)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        hf = m(pixel_values=x).pooler_output.float().cpu()
    pooled, _ = eng(img.to(DEV))
    torch.cuda.synchronize()
    rep = R.cosine_report(pooled.float().cpu(), hf)
    assert rep["cos_min"] >= 0.999 and rep["cos_centered_min"] >= 0.995, rep


def test_profile_accumulates_over_forwards_and_clears_on_read():
    """bench.py's roofline: per-launch CUDA events are kept across the forwards of the timed region and read once."""
    from oracle import siglip_ref as R

    eng, _ = _engine("tiny-hd64", 4)
    img = R.synthetic_images(3, R.CONFIGS["tiny-hd64"].image_size, 0).to(DEV)
    eng.profile(1)
    eng(img)
    one = eng.profile_read()
    assert one["gemm"][1] > 0 and one["attention"][1] > 0 and one["gemm"][0] > 0.0
    assert sum(v[1] for v in eng.profile_read().values()) == 0, "a read clears the record"
    eng.profile(3)
    for _ in range(3):
        eng(img)
    three = eng.profile_read()
    assert {k: v[1] for k, v in three.items()} == {k: 3 * v[1] for k, v in one.items()}
    eng.profile(1)  # room for one forward (16 + 8 L launches): later launches are dropped, never written out of bounds
    for _ in range(4):
        eng(img)
    assert sum(v[1] for v in eng.profile_read().values()) <= 16 + 8 * R.CONFIGS["tiny-hd64"].num_hidden_layers
    eng.profile(0)
    eng(img)
    assert sum(v[1] for v in eng.profile_read().values()) == 0
    eng.close()


@pytest.mark.parametrize("fuse_ln", [False, True])
def test_cuda_graph_replay_is_bit_equal_to_eager(fuse_ln):
    """dfd_engine_set_graphs: a call signature runs eagerly once, is captured on its second sight and replayed afterwards; the
    replays (one cudaGraphLaunch instead of 7·L + 13 launches) give the eager result bit for bit, also on the legacy default
    stream (capture happens on a private stream), for new pixel values in the same buffer, for a second batch size, and the
    launch counter keeps counting the kernels a replay stands for."""
    from dfd import _lib, engine
    from oracle import siglip_ref as R

    name = "tiny-hd72"
    c = R.CONFIGS[name]
    sd = R.init_state_dict(c, 0)
    eager = engine.SiglipEngine(engine.ARCHS[name], 0, max_batch=8, fuse_ln=fuse_ln).load_state_dict(sd)
    graph = engine.SiglipEngine(engine.ARCHS[name], 0, max_batch=8, fuse_ln=fuse_ln, graphs=True).load_state_dict(sd)
    lib = _lib.load()
    buf = {B: torch.empty((B, c.image_size, c.image_size, 3), dtype=torch.uint8, device=DEV) for B in (3, 6)}
    per_forward = None
    for it in range(5):
        for B in (3, 6):
            buf[B].copy_(R.synthetic_images(B, c.image_size, 10 * it + B).to(DEV))   # same buffer, new pixels
            ref, ref_last = eager(buf[B], want_last_hidden=True)
            n0 = lib.dfd_launch_count()
            got, got_last = graph(buf[B], want_last_hidden=True)
            n = lib.dfd_launch_count() - n0
            torch.cuda.synchronize()
            assert torch.equal(ref, got) and torch.equal(ref_last, got_last), (it, B)
            per_forward = per_forward or n
            assert n == per_forward, "a replay accounts for the same number of kernel launches as an eager forward"
    # per batch size: 1 eager run, 1 capture + launch, 3 replays
    assert graph.graph_replays == 2 * 4
    assert eager.graph_replays == 0
    with torch.cuda.stream(torch.cuda.Stream()):     # a non-default stream is a new launch target, not a new signature
        got2, _ = graph(buf[3], want_last_hidden=True)
    torch.cuda.synchronize()
    assert torch.equal(got2, eager(buf[3])[0]) and graph.graph_replays == 9
    graph.set_graphs(False)
    assert torch.equal(graph(buf[6])[0], eager(buf[6])[0]) and graph.graph_replays == 9
    eager.close()
    graph.close()


def test_bench_dump_outputs_are_the_last_steps_records(tmp_path):
    """bench.py --dump-outputs: one float32 .npy per field of the last timed step's score records.  Each field equals what
    DetectionPipeline.detect_device returns for the bench's seeded weights and images (bench.seeded_workload, run here in
    process), for runs with 1 and 3 timed steps; the JSON line reports the requested number of timed steps."""
    import importlib.util
    import json
    import os
    import subprocess
    import sys

    import numpy as np

    from dfd import pipeline
    from dfd.engine import ARCHS

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    names = list(pipeline.PACKED_FIELDS[:pipeline.PACKED_FIELDS.index("risk_p0")]) + ["risk_probs"]
    B, arch_name = 16, bench.WORKLOADS["base-224"][0]
    pipe, images = bench.seeded_workload(ARCHS[arch_name], B, 0, max_batch=B)
    out = pipe.detect_device(images, None, clahe=True)
    want = {n: out[n].float().cpu().numpy() for n in names}
    pipe.engine.close()
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "base-224", "--batch", str(B),
                            "--steps", str(steps), "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in names)
        for n in names:
            got = np.load(d / (n + ".npy"))
            assert got.dtype == np.float32 and got.shape == want[n].shape, (n, got.dtype, got.shape)
            # the frequency features sum per-CTA partials with a double-precision atomicAdd: allow last-bit differences
            assert np.allclose(got, want[n], rtol=1e-5, atol=1e-6), (n, float(np.abs(got - want[n]).max()))
        assert np.array_equal(np.load(d / "risk_idx.npy"), want["risk_idx"])

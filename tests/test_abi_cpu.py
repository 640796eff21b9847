"""CPU tests (no GPU): the C-ABI library builds, loads and exports every symbol include/dfd.h declares, the
ctypes structs mirror the C structs, argument validation works without a device, and compute entry points
FAIL LOUDLY (no CPU fallback) when there is no GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from dfd import _lib

    if not _lib.LIB_PATH.exists():
        import __graft_entry__ as g

        g.build()
    return _lib.load()


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "dfd.h")).read()
    return sorted(set(re.findall(r"DFD_API\s+[\w\s\*]+?\b(dfd_\w+)\s*\(", txt)))


def test_header_symbols_exported(lib):
    from dfd import _lib

    names = _declared_symbols()
    assert len(names) >= 20
    out = subprocess.run(["nm", "-D", "--defined-only", str(_lib.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (dfd_\w+)", out))
    for n in names:
        assert n in exported, f"{n} declared in include/dfd.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert exported - set(_lib.SIGNATURES) == set(), "exported symbol without a binding"


def test_struct_layouts_match_c(tmp_path):
    """sizeof() of every struct crossing the ABI, as the C compiler sees it, equals the ctypes mirror."""
    from dfd import _lib

    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "dfd.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                   "sizeof(dfd_gemm_epilogue),sizeof(dfd_head_weights),sizeof(dfd_score_weights),sizeof(dfd_scores),"
                   "sizeof(dfd_config));return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    sizes = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    assert sizes == [C.sizeof(_lib.GemmEpilogue), C.sizeof(_lib.HeadWeights), C.sizeof(_lib.ScoreWeights),
                     C.sizeof(_lib.Scores), C.sizeof(_lib.EngineConfig)]


def test_version_and_error_text(lib):
    assert lib.dfd_version() >= 100
    assert lib.dfd_launch_count() >= 0
    rc = lib.dfd_gemm_bf16(None, 0, None, 0, None, 0, 1, 1, 1, None, None)
    assert rc == -1 and b"null" in lib.dfd_last_error()
    # per image: half spectrum + counters + 4 column-pass partial slots (freq.cu kImgScratch)
    assert lib.dfd_freq_scratch_bytes(3) == 3 * (256 * 129 * 8 + 272 + 8 * 2048)
    assert lib.dfd_freq_scratch_bytes(0) == 0
    assert lib.dfd_engine_destroy(None) == 0 and lib.dfd_engine_workspace_bytes(None) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
def test_no_cpu_fallback_without_device(lib):
    from dfd import _lib, engine

    cfg = _lib.EngineConfig(64, 16, 128, 256, 2, 2, 1, 1e-6, 0)
    h = C.c_void_p()
    rc = lib.dfd_engine_create(C.byref(cfg), 0, 4, C.byref(h))
    assert rc in (-4, -5) and not h.value, lib.dfd_last_error()
    with pytest.raises(RuntimeError):
        engine.SiglipEngine(engine.ARCHS["tiny-hd64"], 0, 4)
    # a GEMM with plausible (host) pointers must not compute anything on the CPU: it reports the missing driver
    buf = (C.c_uint16 * (128 * 64))()
    rc = lib.dfd_gemm_bf16(C.addressof(buf), 64, C.addressof(buf), 64, C.addressof(buf), 64, 128, 64, 64, None, None)
    assert rc in (-4, -5), lib.dfd_last_error()


def test_engine_config_validation(lib):
    from dfd import _lib

    h = C.c_void_p()
    bad = _lib.EngineConfig(64, 16, 130, 256, 2, 2, 1, 1e-6, 0)  # head dim 65
    assert lib.dfd_engine_create(C.byref(bad), 0, 4, C.byref(h)) == -3
    bad = _lib.EngineConfig(64, 16, 128, 256, 2, 3, 1, 1e-6, 0)  # hidden % heads
    assert lib.dfd_engine_create(C.byref(bad), 0, 4, C.byref(h)) == -2
    assert lib.dfd_engine_create(None, 0, 4, C.byref(h)) == -1


def test_state_dict_canonicalisation_hf_and_timm():
    """HF split q/k/v and timm fused qkv / attn_pool layouts land on the same canonical names (SURVEY App. B)."""
    from dfd import engine
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd64"]
    sd = R.init_state_dict(c, 0)
    hf = {"vision_model." + k: v for k, v in sd.items()}
    canon = engine.canonicalize_state_dict(hf)
    assert set(canon) == set(sd)
    D = c.hidden_size
    timm = {"backbone.visual.trunk.patch_embed.proj.weight": sd["embeddings.patch_embedding.weight"],
            "backbone.visual.trunk.patch_embed.proj.bias": sd["embeddings.patch_embedding.bias"],
            "backbone.visual.trunk.pos_embed": sd["embeddings.position_embedding.weight"][None],
            "backbone.visual.trunk.norm.weight": sd["post_layernorm.weight"],
            "backbone.visual.trunk.norm.bias": sd["post_layernorm.bias"],
            "backbone.visual.trunk.attn_pool.latent": sd["head.probe"],
            "backbone.visual.trunk.attn_pool.q.weight": sd["head.attention.in_proj_weight"][:D],
            "backbone.visual.trunk.attn_pool.q.bias": sd["head.attention.in_proj_bias"][:D],
            "backbone.visual.trunk.attn_pool.kv.weight": sd["head.attention.in_proj_weight"][D:],
            "backbone.visual.trunk.attn_pool.kv.bias": sd["head.attention.in_proj_bias"][D:],
            "backbone.visual.trunk.attn_pool.proj.weight": sd["head.attention.out_proj.weight"],
            "backbone.visual.trunk.attn_pool.proj.bias": sd["head.attention.out_proj.bias"],
            "backbone.visual.trunk.attn_pool.norm.weight": sd["head.layernorm.weight"],
            "backbone.visual.trunk.attn_pool.norm.bias": sd["head.layernorm.bias"],
            "backbone.text.transformer.whatever": torch.zeros(3), "backbone.logit_scale": torch.zeros(())}
    for nm in ("fc1", "fc2"):
        for wb in ("weight", "bias"):
            timm[f"backbone.visual.trunk.attn_pool.mlp.{nm}.{wb}"] = sd[f"head.mlp.{nm}.{wb}"]
    for i in range(c.num_hidden_layers):
        p, t = f"encoder.layers.{i}.", f"backbone.visual.trunk.blocks.{i}."
        for wb in ("weight", "bias"):
            timm[t + "attn.qkv." + wb] = torch.cat([sd[p + f"self_attn.{n}_proj.{wb}"] for n in "qkv"], 0)
            timm[t + "attn.proj." + wb] = sd[p + "self_attn.out_proj." + wb]
            for a, b in (("norm1", "layer_norm1"), ("norm2", "layer_norm2"), ("mlp.fc1", "mlp.fc1"), ("mlp.fc2", "mlp.fc2")):
                timm[t + a + "." + wb] = sd[p + b + "." + wb]
    ct = engine.canonicalize_state_dict(timm)
    assert "head.attention.in_proj_weight" in ct and torch.equal(ct["head.attention.in_proj_weight"], sd["head.attention.in_proj_weight"])
    assert torch.equal(ct["encoder.layers.1.self_attn.qkv.weight"][D:2 * D], sd["encoder.layers.1.self_attn.k_proj.weight"])
    assert not any("text" in k or "logit_scale" in k for k in ct)
    a = engine.arch_from_state_dict(hf)
    assert (a.image_size, a.patch_size, a.hidden_size, a.intermediate_size, a.num_hidden_layers, a.num_attention_heads) == (64, 16, 128, 256, 2, 2)
    assert abs(engine.ARCHS["google/siglip2-so400m-patch14-384"].flops_per_image() / 1e9 - 670.346) < 1e-3


@pytest.mark.parametrize("num_m,num_n,units", [(1458, 14, 74), (1458, 5, 74), (1458, 17, 74), (196, 3, 74), (196, 9, 74),
                                               (3, 2, 148), (1, 1, 148), (7, 5, 5), (50, 4, 6), (371, 5, 74)])
def test_gemm_schedule_takes_every_tile_once_and_balances_the_tail(lib, num_m, num_n, units):
    """The GEMM kernel's persistent schedule, through the same function the kernel uses: every tile exactly once, each
    round a contiguous block of tiles (so concurrent units share A row blocks), and the tail n-tile spread over ALL units
    (a fixed assignment pinned it to the units with (u + r U) mod num_n == num_n - 1: odd units only for 74 / 14)."""
    num_tiles = num_m * num_n
    units = min(units, num_tiles)
    rounds = (num_tiles + units - 1) // units
    seen, tails = [], [0] * units
    for r in range(rounds + 1):
        got = [lib.dfd_gemm_schedule(num_tiles, num_n, units, u, r) for u in range(units)]
        real = sorted(t for t in got if t >= 0)
        if r < rounds:
            assert real == list(range(r * units, min((r + 1) * units, num_tiles))), r
        else:
            assert real == []
        for u, t in enumerate(got):
            if t >= 0 and t % num_n == num_n - 1:
                tails[u] += 1
        seen += real
    assert sorted(seen) == list(range(num_tiles))
    if rounds >= 4 * num_n and num_n > 1:  # long enough for the rotation to show: no unit is starved of / pinned to tail tiles
        assert min(tails) >= 1 and max(tails) <= 2 * (sum(tails) / units) + 1, (min(tails), max(tails))
    assert lib.dfd_gemm_schedule(num_tiles, num_n, units, units, 0) == -1 and lib.dfd_gemm_schedule(0, 1, 1, 0, 0) == -1


def test_freq_luts_equal_oracle_tables():
    import numpy as np

    from dfd import scoring
    from oracle import scoring_ref as S

    band, rbin, sector = scoring.build_freq_tables()
    b, r, s = S.grid_tables()
    assert np.array_equal(band.numpy(), b) and np.array_equal(rbin.numpy(), r) and np.array_equal(sector.numpy(), s)
    # the packed device table: transposed words, then the bin populations the kernel divides by
    lut = scoring.build_freq_luts("cpu").numpy()
    assert lut.shape == (256 * 256 + 48,) and lut.dtype == np.int32
    w = lut[: 256 * 256].reshape(256, 256).T
    assert np.array_equal(w & 0xFF, b) and np.array_equal(((w >> 8) & 0xFF).astype(np.uint8).view(np.int8), r)
    assert np.array_equal(((w >> 16) & 0xFF).astype(np.uint8).view(np.int8), s)
    assert [int(v) for v in lut[256 * 256: 256 * 256 + 40]] == [int((r == i).sum()) for i in range(40)]
    assert [int(v) for v in lut[256 * 256 + 40:]] == [int((s == i).sum()) for i in range(8)]


def test_coral_loader_formats(tmp_path, shipped):
    import json

    from dfd import scoring

    c, t = scoring.load_coral(os.path.join(shipped["dir"], "coral_cutpoints.json"), os.path.join(shipped["dir"], "coral_temp.json"))
    assert abs(c[0] + 1.14372) < 1e-5 and abs(t - 0.9956228137016296) < 1e-12
    (tmp_path / "c.json").write_text(json.dumps([-2.0, -0.5, 0.5, 1.5]))
    (tmp_path / "t.json").write_text("1.7")
    c, t = scoring.load_coral(str(tmp_path / "c.json"), str(tmp_path / "t.json"))
    assert c == [-2.0, -0.5, 0.5, 1.5] and t == 1.7
    (tmp_path / "t2.json").write_text(json.dumps({"temp": 0.8}))
    assert scoring.load_coral(None, str(tmp_path / "t2.json"))[1] == 0.8
    assert abs(scoring.load_coral(None, None)[0][0] - scoring._logit(0.32)) < 1e-12
    # coral.py-style writer round-trips through the loader
    rng = __import__("numpy").random.default_rng(0)
    lg = rng.normal(0, 2, 501).astype("float32")
    art = scoring.write_coral_artifacts(str(tmp_path / "coral"), lg)
    c2, t2 = scoring.load_coral(str(tmp_path / "coral_cutpoints.json"), str(tmp_path / "coral_temp.json"))
    assert c2 == art["cutpoints"] == scoring.fit_coral_cutpoints(lg) and t2 == 1.0
    assert __import__("numpy").load(str(tmp_path / "coral_bins.npy")).sum() == 501
    assert scoring.fit_coral_cutpoints_shipped(shipped["bins"]) == {k: float(shipped["cuts"][k]) for k in ("q25", "q50", "q75", "max")}


def test_resample_tables_host_equal_oracle(lib):
    """dfd_resample_coeffs_host is pure host code (double precision, Pillow's precompute_coeffs): no GPU needed."""
    from dfd import ops
    from oracle import gray_ref as G

    for n in (384, 224, 256, 451, 97, 1024, 33, 7, 3000):
        got, want = ops.resample_coeffs(n, 256), G.resample_coeffs(n, 256)
        assert all(np.array_equal(a, b) for a, b in zip(got, want)), n
    for n, m in ((640, 384), (224, 384), (37, 224), (1920, 384)):
        for f in ("bilinear", "bicubic"):
            got, want = ops.resample_coeffs(n, m, f), G.resample_coeffs(n, m, f)
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), (n, m, f)
    # the identity case reproduces the input exactly: one tap of weight 2^22
    xmin, cnt, kk = ops.resample_coeffs(256, 256)
    assert np.array_equal(kk.sum(1), np.full(256, 1 << 22)) and int((kk != 0).sum()) == 256


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the arm the driver times next to ours) on the CPU-runnable config: one JSON line with the
    keys of the bench contract; the CPU sample is described and nothing pretends to have run on a GPU."""
    import json
    import sys

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "base-224",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and "images per step" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "base-224" in line["config"]["workload"]


def test_pipeline_host_helpers_without_a_device():
    """Host-side pieces of DetectionPipeline that need no GPU: the packed score record layout that is all-gathered across
    ranks, and the six multicrop views / weights of detect_core (deepfake-detector-v2/app.py:1418-1430)."""
    from PIL import Image

    from dfd import pipeline
    from dfd.engine import ARCHS

    B = 5
    out = {k: torch.arange(B, dtype=torch.float32) + 10 * i for i, k in enumerate(pipeline.PACKED_FIELDS[:8])}
    out["risk_idx"] = torch.arange(B, dtype=torch.int32) % 5
    out["risk_probs"] = torch.rand(B, 5)
    rec = pipeline.DetectionPipeline.pack(out)
    assert rec.shape == (B, 14) and rec.dtype == torch.float32
    for i, k in enumerate(pipeline.PACKED_FIELDS[:8]):
        assert torch.equal(rec[:, i], out[k]), k
    assert torch.equal(rec[:, 8], out["risk_idx"].float()) and torch.equal(rec[:, 9:], out["risk_probs"])

    p = object.__new__(pipeline.DetectionPipeline)  # no engine: make_multicrops only needs the architecture
    p.arch = ARCHS["siglip2-base-patch16-224"]
    views = p.make_multicrops(Image.new("RGB", (301, 200), (10, 20, 30)))
    assert [v.size for v in views] == [(301, 200), (224, 224), (150, 100), (151, 100), (150, 100), (151, 100)]
    assert len(pipeline.DetectionPipeline.MULTICROP_WEIGHTS) == 6 and abs(sum(pipeline.DetectionPipeline.MULTICROP_WEIGHTS) - 1.0) < 1e-12


def test_decode_only_loader_and_strong_scaling_unit_plan(tmp_path):
    """Host-side pieces of the device-preprocess path (no GPU): `decode_only` + `ragged_collate` hand the DataLoader's samples over
    as a list of u8 HWC tensors of their decoded sizes (inference_ai_human_images.py:155-192 without the host Resize), rows without
    a file are dropped like the reference does; and bench.py's work-queue plan covers every image exactly once for weak and strong
    scaling shapes."""
    import importlib.util

    from PIL import Image

    from dfd import dropin

    rng = np.random.default_rng(0)
    rows, sizes = [], [(40, 50), (64, 64), (33, 71)]
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(tmp_path / f"i{i}.png")
        rows.append(f"i{i}.png,{i % 2}")
    rows.append("gone.png,1")
    (tmp_path / "meta.csv").write_text("file_name,label\n" + "\n".join(rows) + "\n")
    ds = dropin.AIHumanDataset(tmp_path, tmp_path / "meta.csv", transform=dropin.decode_only)
    assert len(ds) == 3
    ld = torch.utils.data.DataLoader(ds, batch_size=2, shuffle=False, collate_fn=dropin.ragged_collate)
    batches = list(ld)
    assert [len(b[0]) for b in batches] == [2, 1] and batches[0][1].tolist() == [0, 1] and batches[1][2] == ["i2.png"]
    got = [tuple(t.shape) for b in batches for t in b[0]]
    assert got == [(h, w, 3) for h, w in sizes] and all(t.dtype == torch.uint8 for b in batches for t in b[0])
    with Image.open(tmp_path / "i2.png") as pil:
        assert np.array_equal(batches[1][0][0].numpy(), np.asarray(pil.convert("RGB")))

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for total, world, B, sub in [(5 * 512, 1, 512, 512), (5 * 4096, 8, 512, 256), (10 * 512, 8, 64, 64), (10 * 512, 2, 256, 256),
                                 (3 * 96, 4, 24, 12)]:
        plan = bench.unit_plan(total, world, B, sub)
        assert plan[0][0] == 0 and sum(n for _, n in plan) == total
        assert all(plan[i][0] + plan[i][1] == plan[i + 1][0] for i in range(len(plan) - 1))    # contiguous, no overlap
        assert all(0 < n <= sub for _, n in plan)
        if world > 1 and sub % 4 == 0:
            assert plan[-1][1] <= sub // 4          # the queue ends in quarter-size units


def test_fused_normalise_rounds_to_the_reference_bf16_for_every_byte():
    """patchify_u8_rows_kernel computes ToTensor + Normalize(.5,.5) as ONE fp32 FMA, fmaf(x, 2/255, -1); the reference chain is
    ((x / 255) - 0.5) / 0.5 with three fp32 roundings (inference_ai_human_images.py:200-204).  The two differ by an ulp for most
    bytes but round to the same bf16 for all 256 of them — the exhaustive check behind the kernel's comment."""
    x = np.arange(256, dtype=np.float32)
    ref = ((x / np.float32(255.0)) - np.float32(0.5)) / np.float32(0.5)
    fma = (x.astype(np.float64) * np.float64(np.float32(2.0 / 255.0)) - 1.0).astype(np.float32)   # one rounding, like fmaf
    assert torch.equal(torch.from_numpy(ref).to(torch.bfloat16), torch.from_numpy(fma).to(torch.bfloat16))
    tt = torch.arange(256, dtype=torch.uint8).reshape(1, 256, 1).numpy()
    from torchvision import transforms
    tv = transforms.Normalize([0.5], [0.5])(transforms.ToTensor()(tt.transpose(1, 2, 0))).reshape(-1)
    assert torch.equal(tv.to(torch.bfloat16), torch.from_numpy(fma).to(torch.bfloat16))


def test_tiled_layout_of_the_low_halves_round_trips():
    """ops.lo_to_tiled / lo_from_tiled: the [row block][64-column chunk][8-column group][row][8] order the GEMM epilogue and
    dfd_layernorm_bf16 address (element (r, c) at (((r/128·nch + c/64)·8 + (c%64)/8)·128 + r%128)·8 + c%8)."""
    import torch

    from dfd import ops

    for M, N in ((300, 200), (128, 64), (1, 8), (777, 1152)):
        lo = torch.randn(M, N).to(torch.bfloat16)
        t = ops.lo_to_tiled(lo)
        nch = (N + 63) // 64
        assert tuple(t.shape) == ((M + 127) // 128, nch, 8, 128, 8)
        assert torch.equal(ops.lo_from_tiled(t, M, N), lo)
        flat = t.reshape(-1)
        for r, c in ((0, 0), (M - 1, N - 1), (M // 2, N // 3), (min(M - 1, 129), min(N - 1, 70))):
            idx = (((r // 128 * nch + c // 64) * 8 + (c % 64) // 8) * 128 + r % 128) * 8 + c % 8
            assert flat[idx] == lo[r, c], (M, N, r, c)

"""GPU tests of the reference-shaped Python surface (dfd.dropin, dfd.pipeline, dfd.train_fusion) against the oracle."""
import os

import numpy as np
import pytest
import torch

from tests.reference_style import reference_style_classifier

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bc(head, name="tiny-hd64"):
    from dfd import dropin
    from oracle import siglip_ref as R

    c = R.CONFIGS[name]
    sd = R.init_state_dict(c, 0)
    hs = R.init_head(head, c.hidden_size, 1)
    m = dropin.BinaryClassifier(device=DEV, head=head, arch=name, max_batch=8)
    ck = {"backbone.vision_model." + k: v for k, v in sd.items()}
    ck.update(hs)
    ck["backbone.text.whatever"] = torch.zeros(4)
    m.load_state_dict(ck, strict=True)
    return m, c, sd, hs


@pytest.mark.parametrize("head,eps", [("A", 0.0), ("B", 1e-6)])
def test_binary_classifier_forward(head, eps):
    from oracle import siglip_ref as R

    m, c, sd, hs = _bc(head)
    assert m.resolution == c.image_size and set(m.classifier.state_dict()) >= {"0.weight", "2.weight", "5.weight"}
    x = R.preprocess_u8(R.synthetic_images(5, c.image_size, 3))
    z = m(x).cpu()
    pooled = R.siglip_vision_forward(sd, c, x, "fp32")["pooler_output"]
    z_ref = R.classifier_head(hs, head, pooled, eps)
    # 128-wide toy model with the production engine mode (LayerNorm folded into the GEMMs): bf16 noise averages over 6-9x
    # fewer channels than at the named architectures, where the 1e-2 gate is asserted (tests/test_engine_gpu.py:
    # test_benched_configuration_vs_hf_on_gpu, test_base_224_logits) — 2e-2 here, as for the other toy-model checks
    assert (z - z_ref).abs().max() < 2e-2 * max(1.0, float(z_ref.abs().max())), (z, z_ref)
    if head == "B":  # off-size input -> F.interpolate default (nearest) inside the model
        xs = R.preprocess_u8(R.synthetic_images(3, 40, 4))
        z2 = m(xs).cpu()
        p2 = R.siglip_vision_forward(sd, c, R.resize_input(xs, c.image_size, "nearest"), "fp32")["pooler_output"]
        assert (z2 - R.classifier_head(hs, "B", p2, 1e-6)).abs().max() < 2e-2


def test_fast_binary_classifier_cifake_path():
    """BASELINE config 4: 32x32 images, bilinear align_corners=False upsampling inside the model, head H-D."""
    from dfd import dropin
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd64"]
    sd = R.init_state_dict(c, 0)
    for size in ("small", "large"):
        hd = R.init_head_d(size, c.hidden_size, 4)
        m = dropin.FastBinaryClassifier(size, DEV, arch="tiny-hd64", max_batch=8)
        ck = {"backbone.vision_model." + k: v for k, v in sd.items()}
        ck.update(hd)
        m.load_state_dict(ck)
        img = R.synthetic_images(7, 32, 8)
        for x in (img, R.preprocess_u8(img)):  # u8 NHWC and normalised f32 NCHW
            z = m(x).cpu()
            xr = R.resize_input(R.preprocess_u8(img), c.image_size, "bilinear")
            z_ref = R.classifier_head_d(hd, R.siglip_vision_forward(sd, c, xr, "fp32")["pooler_output"])
            assert (z - z_ref).abs().max() < 2e-2 * max(1.0, float(z_ref.abs().max())), (size, z, z_ref)


def test_run_inference_and_prototypes():
    from dfd import dropin
    from oracle import siglip_ref as R

    m, c, sd, hs = _bc("A")
    imgs = R.preprocess_u8(R.synthetic_images(12, c.image_size, 5))
    labels = torch.tensor([0, 1] * 6)
    loader = [(imgs[i:i + 4], labels[i:i + 4], [f"f{j}.png" for j in range(i, i + 4)]) for i in range(0, 12, 4)]
    lab, probs, files = dropin.run_inference(m, loader, torch.device(DEV))
    pooled = R.siglip_vision_forward(sd, c, imgs, "fp32")["pooler_output"]
    p_ref = torch.sigmoid(R.classifier_head(hs, "A", pooled, 0.0)).numpy()
    assert lab.tolist() == labels.tolist() and files[5] == "f5.png"
    assert np.abs(probs - p_ref).max() < 5e-3
    _, pinv, _ = dropin.run_inference(m, loader, torch.device(DEV), invert_logits=True)
    assert np.abs(pinv - (1 - p_ref)).max() < 5e-3
    protos = dropin.few_shot_prototype(m, loader, torch.device(DEV))
    f = R.l2_normalize(pooled)
    pr = torch.stack([f[labels == 0].mean(0), f[labels == 1].mean(0)])
    pr = pr / pr.norm(dim=-1, keepdim=True)
    assert (protos["real"].cpu() - pr[0]).abs().max() < 5e-3 and (protos["fake"].cpu() - pr[1]).abs().max() < 5e-3
    _, pp, _ = dropin.run_inference(m, loader, torch.device(DEV), prototypes=protos)
    pp_ref = R.prototype_prob(f, protos["real"].cpu(), protos["fake"].cpu()).numpy()
    assert np.abs(pp - pp_ref).max() < 5e-3


def test_hf_shaped_vision_model():
    from dfd import dropin
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd72"]
    sd = R.init_state_dict(c, 0)
    m = dropin.SiglipVisionModel.from_state_dict({"vision_model." + k: v for k, v in sd.items()}, DEV, num_heads=2)
    assert m.config.hidden_size == c.hidden_size
    x = R.preprocess_u8(R.synthetic_images(2, c.image_size, 0))
    o = m(pixel_values=x)
    ref = R.siglip_vision_forward(sd, c, x, "fp32")
    assert R.cosine_report(o.pooler_output.cpu(), ref["pooler_output"])["cos_min"] >= 0.999
    assert o.last_hidden_state.shape == (2, c.tokens, c.hidden_size)
    # per-layer hidden states (SigLIP2_MTL taps, Siglip2sidafrozen.py:787-793)
    oh = m(pixel_values=x, output_hidden_states=True)
    rh = R.siglip_vision_forward(sd, c, x, "fp32", output_hidden_states=True)["hidden_states"]
    assert len(oh.hidden_states) == c.num_hidden_layers + 1 == len(rh)
    for a, b in zip(oh.hidden_states, rh):
        rep = R.cosine_report(a.cpu().reshape(-1, c.hidden_size), b.reshape(-1, c.hidden_size))
        assert rep["cos_min"] >= 0.998 and rep["rel_l2"] <= 0.03, rep
    assert torch.equal(oh.pooler_output, o.pooler_output)


def test_import_shims():
    from dfd import dropin
    from oracle import scoring_ref as S

    dropin.install_import_shims()
    import open_clip
    import pywt

    model, _, pre = open_clip.create_model_and_transforms("tiny-hd64", pretrained="webli", device=DEV)
    assert model.embed_dim == 128 and callable(pre)
    from PIL import Image

    t = pre(Image.fromarray(np.zeros((50, 70, 3), np.uint8)))
    assert t.shape == (3, 64, 64) and float(t.max()) == -1.0
    x = np.random.default_rng(0).random((16, 16)).astype(np.float32)
    cA, (cH, cV, cD) = pywt.dwt2(x, "db1")
    for a, b in zip((cA, cH, cV, cD), S.haar2(x)):
        assert np.array_equal(a, b)


def test_detection_pipeline_host_buffers_vs_oracle():
    """The public e2e call (pinned host buffers in, packed score records out) against the oracle stack."""
    from dfd import pipeline, scoring
    from oracle import scoring_ref as S
    from oracle import siglip_ref as R

    name = "tiny-hd72"
    c = R.CONFIGS[name]
    sd, hs = R.init_state_dict(c, 0), R.init_head("B", c.hidden_size, 1)
    cuts = [-1.0, -0.2, 0.3, 1.5]
    st = scoring.ScoringStack(DEV, S.init_freq_mlp_g2(2), S.init_fusion_g2(3), cuts, 1.1)
    pipe = pipeline.DetectionPipeline(name, sd, hs, st, device=0, max_batch=4)
    img = R.synthetic_images(6, c.image_size, 7)
    gray = np.stack([S.gray256_from_rgb_u8(im.numpy(), True) for im in img])
    rec = pipe.detect(img.pin_memory(), torch.from_numpy(gray).pin_memory())
    assert rec.shape == (6, len(pipeline.PACKED_FIELDS))
    col = {k: i for i, k in enumerate(pipeline.PACKED_FIELDS)}
    pooled = R.siglip_vision_forward(sd, c, R.preprocess_u8(img), "fp32")["pooler_output"]
    z_sig = R.classifier_head(hs, "B", pooled, 1e-6).numpy()
    feats = np.stack([S.extract_freq_vector(g) for g in gray])
    z_freq = S.freq_mlp_g2(S.init_freq_mlp_g2(2), feats)
    z = S.fusion_g2(S.init_fusion_g2(3), z_freq, z_sig)
    d = S.detect_scores(z, np.array(cuts, np.float32), 1.1)
    # Logit gate.  BASELINE asks for 1e-2 at the named (768/1152-wide) architectures — checked in
    # tests/test_engine_gpu.py::test_base_224_logits.  On this 144-wide toy model bf16 noise averages over 5-8x fewer
    # channels: the reference's own bf16-autocast path is already up to 8e-3 from fp32 here, so the bound is 2e-2
    # (max) with the median held at 5e-3.
    pooled_ac = R.siglip_vision_forward(sd, c, R.preprocess_u8(img), "autocast")["pooler_output"]
    z_sig_ac = R.classifier_head(hs, "B", pooled_ac, 1e-6).numpy()
    for zr in (z_sig, z_sig_ac):
        e = np.abs(rec[:, col["z_sig"]] - zr)
        assert e.max() < 2e-2 and np.median(e) < 5e-3, e
    assert np.abs(rec[:, col["z_freq"]] - z_freq).max() < 1e-3
    assert np.abs(rec[:, col["z"]] - z).max() < 2e-2
    assert np.abs(rec[:, col["p_blend"]] - d["p_blend"]).max() < 5e-3
    tp = S.coral_transition_points(np.array(cuts, np.float32))
    near = np.abs(d["z_scaled"][:, None] - tp[None]).min(1) < 1e-2
    assert np.array_equal(rec[:, col["risk_idx"]].astype(int)[~near], d["risk_idx"][~near])


def test_detect_core_multicrop_vs_oracle():
    """`detect_core(pil, multicrop=True)` for a batch of images in one call vs the reference flow restated with the
    oracle: 6 crops, weights on logits, G1 shipped heads (z-scored features), temperature, CORAL."""
    from PIL import Image

    from dfd import dropin, pipeline, scoring
    from oracle import scoring_ref as S
    from oracle import siglip_ref as R
    from tests.conftest import SIGLIP_ARTEFACTS

    name = "tiny-hd64"
    c = R.CONFIGS[name]
    sd, hs = R.init_state_dict(c, 0), R.init_head("B", c.hidden_size, 1)
    st = scoring.ScoringStack.from_dir(SIGLIP_ARTEFACTS, DEV)
    pipe = pipeline.DetectionPipeline(name, sd, hs, st, device=0, max_batch=16)
    rng = np.random.default_rng(3)
    pils = [Image.fromarray(np.clip(rng.normal(120, 50, (90 + 20 * i, 130, 3)), 0, 255).astype(np.uint8)) for i in range(2)]
    res = pipe.detect_core(pils, multicrop=True, clahe=False)
    assert len(res) == 2 and set(res[0]) >= {"z_sig", "z_freq", "z_scaled", "p_fake_raw", "p_fake_coral", "p_blend",
                                             "risk_idx", "risk_probs", "entropy", "visual_prob", "freq_prob"}
    import json
    from safetensors.torch import load_file

    fm, fu = load_file(f"{SIGLIP_ARTEFACTS}/freq_mlp.safetensors"), load_file(f"{SIGLIP_ARTEFACTS}/fusion_head.safetensors")
    cuts = S.coral_cut_logits(json.load(open(f"{SIGLIP_ARTEFACTS}/coral_cutpoints.json")))
    temp = json.load(open(f"{SIGLIP_ARTEFACTS}/coral_temp.json"))["temperature"]
    pre = dropin.make_preprocess(c.image_size, "bilinear")
    w = np.array(pipeline.DetectionPipeline.MULTICROP_WEIGHTS)
    for pil, r in zip(pils, res):
        crops = pipe.make_multicrops(pil)
        x = torch.stack([pre(v) for v in crops])
        pooled = R.siglip_vision_forward(sd, c, x, "fp32")["pooler_output"]
        z_sig = float((R.classifier_head(hs, "B", pooled, 1e-6).numpy() * w).sum())
        feats = np.stack([S.extract_freq_vector(S.gray256_from_rgb_u8(np.asarray(v), False), zscore=True) for v in crops])
        z_freq = float((S.freq_mlp_g1(fm, feats) * w).sum())
        z = S.fusion_g1(fu, np.array([z_sig]), np.array([z_freq]))
        d = S.detect_scores(z, cuts, temp)
        assert abs(r["z_sig"] - z_sig) < 2e-2 and abs(r["z_freq"] - z_freq) < 2e-3
        assert abs(r["z_scaled"] - float(d["z_scaled"][0])) < 1e-2 and abs(r["p_blend"] - float(d["p_blend"][0])) < 5e-3
        assert r["risk_idx"] == int(d["risk_idx"][0])
        assert abs(r["visual_prob"] - 1 / (1 + np.exp(-z_sig))) < 5e-3


def _reference_fit(z_freq, z_sig, labels, batch_size, epochs, seed):
    """train_fusion_head_only.py:402-447 restated with torch autograd under enable_grad (SURVEY.md §0.4)."""
    import torch.nn as nn
    import torch.nn.functional as F
    from torch.utils.data import DataLoader, TensorDataset

    class Head(nn.Module):
        def __init__(self):
            super().__init__()
            self.mlp = nn.Sequential(nn.Linear(3, 32), nn.GELU(), nn.Linear(32, 2))
            self.T = nn.Parameter(torch.tensor(1.0))

        def forward(self, zf, zs):
            w = F.softmax(self.mlp(torch.stack([zf, zs, (zf - zs).abs()], -1)), -1)
            return (w[..., 0] * zf + w[..., 1] * zs) / (self.T + 1e-6)

    torch.manual_seed(seed)
    h = Head()
    loader = DataLoader(TensorDataset(torch.stack([z_freq, z_sig], 1), labels), batch_size=batch_size, shuffle=True)
    opt = torch.optim.AdamW(h.parameters(), lr=5e-4)
    with torch.enable_grad():
        for _ in range(epochs):
            for xb, yb in loader:
                opt.zero_grad()
                loss = nn.BCEWithLogitsLoss()(h(xb[:, 0], xb[:, 1]), yb)
                loss.backward()
                nn.utils.clip_grad_norm_(h.parameters(), max_norm=5.0)
                opt.step()
    return torch.cat([p.detach().reshape(-1) for p in (h.mlp[0].weight, h.mlp[0].bias, h.mlp[2].weight, h.mlp[2].bias, h.T)])


def test_fit_fusion_head_matches_reference_loop():
    from dfd import train_fusion

    rng = np.random.default_rng(0)
    n = 203  # ragged last mini-batch
    y = torch.from_numpy((rng.random(n) > 0.5).astype(np.float32))
    zs = torch.from_numpy((rng.normal(0, 2, n) + 2.0 * (y.numpy() - 0.5)).astype(np.float32))
    zf = torch.from_numpy((rng.normal(0, 2, n) + 1.0 * (y.numpy() - 0.5)).astype(np.float32))
    ref = _reference_fit(zf, zs, y, 32, 3, seed=11)
    torch.manual_seed(11)
    head, best, auc = train_fusion.fit_fusion_head(zf, zs, y, batch_size=32, epochs=3, device=DEV, verbose=False)
    got = head.flat.data.cpu()
    assert (got - ref).abs().max() < 2e-4, (got - ref).abs().max()
    assert set(best) == {"mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias", "temp.T"}
    assert tuple(best["mlp.0.weight"].shape) == (32, 3) and best["temp.T"].shape == ()
    assert auc > 0.6


def test_train_fusion_head_end_to_end(tmp_path):
    """Entry point #2 on synthetic image folders: extraction -> training -> fusion_head.safetensors in the
    reference layout, loadable by the G2 scoring stack."""
    from PIL import Image
    from safetensors.torch import load_file, save_file

    from dfd import scoring, train_fusion
    from oracle import scoring_ref as S
    from oracle import siglip_ref as R

    rng = np.random.default_rng(1)
    for cls, shift in (("real", 0), ("fake", 60)):
        os.makedirs(tmp_path / cls)
        for i in range(6):
            arr = np.clip(rng.normal(110 + shift, 40, (48 + 8 * i, 64, 3)), 0, 255).astype(np.uint8)
            Image.fromarray(arr).save(tmp_path / cls / f"{i}.png")
    c = R.CONFIGS["tiny-hd64"]
    ck = {"backbone.vision_model." + k: v.contiguous() for k, v in R.init_state_dict(c, 0).items()}
    ck.update({k: v.contiguous() for k, v in R.init_head("B", c.hidden_size, 1).items()})
    save_file(ck, str(tmp_path / "best_model.safetensors"))
    save_file({k: v.contiguous() for k, v in S.init_freq_mlp_g2(2).items()}, str(tmp_path / "freq_mlp.safetensors"))
    out = tmp_path / "fusion_head.safetensors"
    torch.manual_seed(0)
    best = train_fusion.train_fusion_head(str(tmp_path / "real"), str(tmp_path / "fake"), str(tmp_path / "best_model.safetensors"),
                                          str(tmp_path / "freq_mlp.safetensors"), str(out), batch_size=4, epochs=2,
                                          device=DEV, arch="tiny-hd64")
    sd = load_file(str(out))
    assert {k: tuple(v.shape) for k, v in sd.items()} == {"mlp.0.weight": (32, 3), "mlp.0.bias": (32,), "mlp.2.weight": (2, 32),
                                                        "mlp.2.bias": (2,), "temp.T": ()}
    assert all(torch.equal(sd[k], best[k]) for k in sd)
    st = scoring.ScoringStack(DEV, load_file(str(tmp_path / "freq_mlp.safetensors")), sd, [-1.0, -0.2, 0.3, 1.5], 1.0)
    assert st.gen == 2


def test_extract_logits_device_preprocess_equals_host_chain(tmp_path):
    """Entry point #2's two extraction loops (train_fusion_head_only.py:329-347) with the preprocess on the GPU — per-channel CLAHE,
    PIL Resize, gray256 from one upload per decoded file — against the reference's own host chain (cv2 + PIL + torchvision,
    `on_device=False`): the device kernels are bit-exact, so the logits agree to the last bit for the frequency branch and to
    fp32 round-off of ToTensor / Normalize (folded into one multiply-add in the patch kernel) before bf16 for SigLIP."""
    from PIL import Image
    from safetensors.torch import load_file, save_file  # noqa: F401

    from dfd import scoring, train_fusion
    from dfd.dropin import BinaryClassifier
    from oracle import scoring_ref as S
    from oracle import siglip_ref as R

    rng = np.random.default_rng(4)
    paths = []
    for i, (h, w) in enumerate([(48, 64), (100, 37), (64, 64), (131, 77), (224, 224), (17, 300)]):
        arr = np.clip(rng.normal(120, 50, (h, w, 3)), 0, 255).astype(np.uint8)
        arr[: h // 2, : w // 2] //= 3      # a dark quadrant: CLAHE has something to equalise
        Image.fromarray(arr).save(tmp_path / f"{i}.png")
        paths.append(str(tmp_path / f"{i}.png"))
    c = R.CONFIGS["tiny-hd64"]
    siglip = BinaryClassifier(device=DEV, head="B", arch="tiny-hd64", max_batch=8)
    ck = {"backbone.vision_model." + k: v for k, v in R.init_state_dict(c, 0).items()}
    ck.update(R.init_head("B", c.hidden_size, 1))
    siglip.load_state_dict(ck, strict=False)
    # the preprocessed pixels themselves: u8 on the device == the host chain before ToTensor
    pre_host = train_fusion.make_preprocess(siglip.resolution)
    for p in paths:
        with Image.open(p) as pil:
            host = pre_host(pil.convert("RGB"))                      # f32 [3,S,S] in [-1,1]
        dev = train_fusion.preprocess_on_device(train_fusion._decode_rgb_u8(p), siglip.resolution, siglip.device)
        want_u8 = torch.round((host * 0.5 + 0.5) * 255.0).permute(1, 2, 0).to(torch.uint8)
        assert torch.equal(dev.cpu(), want_u8), p
    z_dev = train_fusion.extract_siglip_logits(siglip, paths, batch_size=4)
    z_host = train_fusion.extract_siglip_logits(siglip, paths, batch_size=4, on_device=False)
    assert z_dev.shape == z_host.shape == (len(paths),)
    assert float((z_dev - z_host).abs().max()) <= 2e-3, (z_dev, z_host)   # same bf16 pixels up to fp32 round-off of the normalise
    fm = scoring.FreqMLP()
    fm.load_state_dict(S.init_freq_mlp_g2(2), strict=True)
    f_dev = train_fusion.extract_freq_logits(fm, paths, DEV, batch_size=4)
    f_host = train_fusion.extract_freq_logits(fm, paths, DEV, batch_size=4, on_device=False)
    assert torch.equal(f_dev, f_host)


def _reference_fit_freq(features, labels, batch_size, epochs, lr, seed):
    """"FreqMLP trainer.py":330-396 restated with torch autograd, dropout off (the only stochastic part)."""
    import torch.nn as nn
    import torch.nn.functional as F
    from torch.utils.data import DataLoader, TensorDataset

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.norm, self.fc1, self.fc2 = nn.LayerNorm(24), nn.Linear(24, 64), nn.Linear(64, 24)

        def forward(self, x):
            return self.fc2(F.gelu(self.fc1(self.norm(x)))) + x

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.alpha, self.beta = nn.Parameter(torch.ones(24)), nn.Parameter(torch.zeros(24))
            self.gates = nn.Parameter(torch.zeros(4))
            self.blocks = nn.ModuleList([Block(), Block()])
            self.head = nn.Linear(24, 1)
            self.T = nn.Parameter(torch.tensor(1.0))

        def forward(self, x, mean, std):
            x = torch.tanh(self.alpha * ((x - mean) / (std + 1e-6)) + self.beta)
            g = torch.sigmoid(self.gates)
            x = torch.cat([c * g[i] for i, c in enumerate(torch.split(x, 6, dim=-1))], dim=-1)
            for b in self.blocks:
                x = b(x)
            return self.head(x).squeeze(-1) / (self.T + 1e-6)

    torch.manual_seed(seed)
    m = Net()
    mean, std = features.mean(0), features.std(0) + 1e-6
    loader = DataLoader(TensorDataset(features, labels), batch_size=batch_size, shuffle=True)
    opt = torch.optim.AdamW(m.parameters(), lr=lr)
    with torch.enable_grad():
        for _ in range(epochs):
            for xb, yb in loader:
                opt.zero_grad()
                nn.BCEWithLogitsLoss()(m(xb, mean, std), yb).backward()
                nn.utils.clip_grad_norm_(m.parameters(), max_norm=5.0)
                opt.step()
    ps = [m.alpha, m.beta, m.gates]
    for b in m.blocks:
        ps += [b.norm.weight, b.norm.bias, b.fc1.weight, b.fc1.bias, b.fc2.weight, b.fc2.bias]
    ps += [m.head.weight, m.head.bias, m.T]
    return torch.cat([p.detach().reshape(-1) for p in ps])


def test_fit_freq_mlp_matches_reference_loop(tmp_path):
    from safetensors.torch import load_file, save_file

    from dfd import scoring, train_freq

    rng = np.random.default_rng(4)
    n = 101  # ragged last mini-batch
    y = torch.from_numpy((rng.random(n) > 0.5).astype(np.float32))
    feats = torch.from_numpy((rng.normal(0.2, 0.7, (n, 24)) + 0.6 * (y.numpy()[:, None] - 0.5)).astype(np.float32))
    ref = _reference_fit_freq(feats, y, 8, 3, 1e-3, seed=5)
    torch.manual_seed(5)
    model, best, auc = train_freq.fit_freq_mlp(feats, y, epochs=3, batch_size=8, lr=1e-3, device=DEV, dropout=0.0,
                                               verbose=False)
    got = model.flat.data.cpu()
    assert (got - ref).abs().max() < 5e-4, (got - ref).abs().max()
    assert auc > 0.6
    # the written file loads, strictly, into the inference-side FreqMLP (the reference's reader: train_fusion_head_only.py:390-392)
    path = str(tmp_path / "freq_mlp.safetensors")
    save_file({k: v.contiguous() for k, v in best.items()}, path)
    fm = scoring.FreqMLP()
    fm.load_state_dict(load_file(path), strict=True)
    z = fm(feats.to(DEV))
    model.load_state_dict(best)
    assert (z - model(feats.to(DEV))).abs().max() < 1e-4


def test_segformer_decoder_matches_reference_golden(golden_decoder):
    """dfd.mtl.SegFormerStrongDecoder vs the reference's own class (fp32) on its golden inputs: bf16 GEMM chain."""
    from dfd import mtl
    from oracle import decoder_ref as D

    g = golden_decoder
    C, K, E, grid, S, B = (int(v) for v in g["dims"])
    dec = mtl.SegFormerStrongDecoder(K, E, DEV).load_state_dict(D.init_decoder_state(C, K, E, 3), prefix="decoder.")
    hs = [torch.from_numpy(h).reshape(B * grid * grid, C).to(DEV, torch.bfloat16) for h in g["hidden"]]
    out = dec(hs, B, grid, S).cpu().numpy()
    ref = g["seg"]
    # five bf16 GEMMs deep; logits of magnitude ~0.35: 1 % of the range
    assert np.abs(out - ref).max() < 0.01 * max(1.0, float(np.abs(ref).max()) / 0.35), np.abs(out - ref).max()
    assert np.corrcoef(out.ravel(), ref.ravel())[0, 1] > 0.9995


def test_siglip2_mtl_end_to_end():
    """SigLIP2_MTL (encoder taps + 3-class head + decoder) vs the fp32 oracle chain at a small architecture."""
    from dfd import mtl
    from oracle import decoder_ref as D
    from oracle import siglip_ref as R

    name = "small-hd72"                      # 210 px, 15 x 15 tokens, hidden 288, 3 layers
    c = R.CONFIGS[name]
    seg_layers, E = (0, 1, -1), 64
    sd = {"encoder.vision_model." + k: v for k, v in R.init_state_dict(c, 0).items()}
    sd.update(D.init_decoder_state(c.hidden_size, len(seg_layers), E, seed=4))
    model = mtl.SigLIP2_MTL(name, 0, max_batch=2, seg_layers=seg_layers, embed_dim=E).load_state_dict(sd)
    img = R.synthetic_images(2, c.image_size, 3)
    cls, seg = model(img.to(DEV))
    o = R.siglip_vision_forward(R.init_state_dict(c, 0), c, R.preprocess_u8(img), "fp32", output_hidden_states=True)
    hs = o["hidden_states"]
    feats = [hs[i + 1 if i >= 0 else len(hs) - 1] for i in seg_layers]
    seg_ref = D.decoder_forward(sd, feats, 15, c.image_size)
    cls_ref = D.cls_head(sd, o["pooler_output"])
    torch.cuda.synchronize()
    assert tuple(seg.shape) == (2, 1, 210, 210) and tuple(cls.shape) == (2, 3)
    assert (cls.cpu() - cls_ref).abs().max() < 2e-2 * max(1.0, float(cls_ref.abs().max()))
    scale = float(seg_ref.abs().max())
    assert (seg.cpu() - seg_ref).abs().max() < 0.03 * max(scale, 0.3), ((seg.cpu() - seg_ref).abs().max(), scale)
    assert np.corrcoef(seg.cpu().numpy().ravel(), seg_ref.numpy().ravel())[0, 1] > 0.999
    # progressive-resize sizes (Siglip2sidafrozen.py:975-987 with interpolate_pos_encoding=True at :787): 280 px = 20 x 20 tokens
    import dataclasses

    from dfd import dropin

    S2, g2 = 280, 20
    img2 = R.synthetic_images(3, S2, 4)      # 3 images through a max_batch-1 engine (workspace scaled to the token count): chunked
    cls2, seg2 = model(img2.to(DEV))
    sd2 = dict(R.init_state_dict(c, 0))
    sd2["embeddings.position_embedding.weight"] = dropin.interpolated_position_table(sd2["embeddings.position_embedding.weight"], g2)
    c2 = dataclasses.replace(c, image_size=S2) if dataclasses.is_dataclass(c) else type(c)(**{**c.__dict__, "image_size": S2})
    o2 = R.siglip_vision_forward(sd2, c2, R.preprocess_u8(img2), "fp32", output_hidden_states=True)
    hs2 = o2["hidden_states"]
    seg_ref2 = D.decoder_forward(sd, [hs2[i + 1 if i >= 0 else len(hs2) - 1] for i in seg_layers], g2, S2)
    assert tuple(seg2.shape) == (3, 1, S2, S2)
    assert (cls2.cpu() - D.cls_head(sd, o2["pooler_output"])).abs().max() < 2e-2 * max(1.0, float(cls_ref.abs().max()))
    assert np.corrcoef(seg2.cpu().numpy().ravel(), seg_ref2.numpy().ravel())[0, 1] > 0.999


# ---------------------------------------------------------------------------------------------------------------------
# The reference's own flow on the GPU, with its two model classes as tests/reference_style.py restates them (checked
# against the reference's source in tests/test_dropin_cpu.py where a checkout is given), driven like its entry points drive them.
# ---------------------------------------------------------------------------------------------------------------------
def _timm_checkpoint(sd, hs):
    """`best_model` checkpoint as the reference's trainers write it: open_clip/timm backbone names + head + text tower."""
    from dfd import dropin
    from dfd.engine import canonicalize_state_dict

    ck = {"backbone." + k: v.clone() for k, v in dropin.timm_state_from_canonical(canonicalize_state_dict(sd)).items()}
    ck.update({k: v.clone() for k, v in hs.items()})
    ck["backbone.logit_scale"], ck["backbone.logit_bias"] = torch.tensor(2.3), torch.tensor(-10.0)
    ck["backbone.text.token_embedding.weight"] = torch.zeros(4, 8)
    return ck


@pytest.mark.parametrize("kind,eps", [("A", 0.0), ("B", 1e-6)])
def test_reference_style_module_strict_load_inference_mode_autocast(kind, eps):
    """Entry-point flow of inference_ai_human_images.py (:836-857 load, :265-309 loop) / train_fusion_head_only.py
    (:118-124, :339-347): nn.Module that owns the tower as `self.backbone`, strict load of a timm-named checkpoint,
    `inference_mode()` + `autocast()`, sigmoid, `.cpu()`.  The logits must match the oracle ON THE CHECKPOINT'S weights
    (and be far from what the tower's initial random weights give)."""
    import warnings

    from dfd import dropin
    from oracle import siglip_ref as R

    dropin.install_import_shims()
    name = "small-hd72"
    c = R.CONFIGS[name]
    sd, hs = R.init_state_dict(c, 0), R.init_head(kind, c.hidden_size, 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = reference_style_classifier(kind, name, c.hidden_size, c.image_size)(DEV).to(DEV)
    assert model.backbone.weights_source == "random"
    x = R.preprocess_u8(R.synthetic_images(6, c.image_size, 3))
    model.eval()
    with torch.inference_mode(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        z_random = model(x.to(DEV)).float().cpu()
    model.load_state_dict(_timm_checkpoint(sd, hs), strict=True)
    assert model.backbone.weights_source == "checkpoint"
    with torch.inference_mode():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            f = model.backbone.encode_image(x.to(DEV))
            assert f.dtype == torch.bfloat16           # the tower honours the autocast dtype like a torch module would
            z = model(x.to(DEV))
        probs = torch.sigmoid(z).float().cpu().numpy()
        assert model.backbone.encode_image(x.to(DEV)).dtype == torch.float32
    pooled = R.siglip_vision_forward(sd, c, x, "fp32")["pooler_output"]
    z_ref = R.classifier_head(hs, kind, pooled, eps)
    # the head runs as torch modules under autocast here (bf16 GEMMs, as in the reference): 3e-2 on O(1) logits
    assert (z.float().cpu() - z_ref).abs().max() < 3e-2 * max(1.0, float(z_ref.abs().max())), (z, z_ref)
    assert np.abs(probs - torch.sigmoid(z_ref).numpy()).max() < 1e-2
    assert (z_random - z_ref).abs().max() > 0.1, "the strict load must have replaced the random backbone"
    # in-place parameter updates reach the engine too (version counters), not only load_state_dict
    with torch.no_grad():
        model.backbone.visual.trunk.pos_embed.mul_(0.0)
    with torch.inference_mode():
        z2 = model(x.to(DEV)).float().cpu()
    sd2 = dict(sd)
    sd2["embeddings.position_embedding.weight"] = torch.zeros_like(sd["embeddings.position_embedding.weight"])
    z2_ref = R.classifier_head(hs, kind, R.siglip_vision_forward(sd2, c, x, "fp32")["pooler_output"], eps)
    assert (z2 - z2_ref).abs().max() < 3e-2 * max(1.0, float(z2_ref.abs().max()))


def test_reference_style_module_survives_torch_compile():
    """inference_ai_human_images.py:868-881 wraps the model in torch.compile; the tower's forward is opaque to dynamo
    (torch.compiler.disable) and keeps running on the dfd engine, the torch head around it is compiled."""
    import warnings

    from dfd import dropin
    from oracle import siglip_ref as R

    dropin.install_import_shims()
    name = "tiny-hd64"
    c = R.CONFIGS[name]
    sd, hs = R.init_state_dict(c, 0), R.init_head("A", c.hidden_size, 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = reference_style_classifier("A", name, c.hidden_size, c.image_size)(DEV).to(DEV).eval()
    model.load_state_dict(_timm_checkpoint(sd, hs), strict=True)
    x = R.preprocess_u8(R.synthetic_images(4, c.image_size, 3)).to(DEV)
    with torch.inference_mode():
        z_eager = model(x).float().cpu()
    try:
        compiled = torch.compile(model)
        with torch.inference_mode():
            z_c = compiled(x).float().cpu()
    except Exception as e:  # the box may lack a working inductor toolchain; the reference itself falls back to eager then
        pytest.skip(f"torch.compile unavailable here: {type(e).__name__}: {str(e)[:80]}")
    assert (z_c - z_eager).abs().max() < 1e-3, (z_c, z_eager)


def test_run_tta_inference_fused_flip_equals_two_host_passes(tmp_path):
    """run_tta_inference (inference_ai_human_images.py:321-360) with the default 2 transforms: the fused pass (mirrored view
    produced by the patch kernel from the resident pixels) equals the reference's way — a second decode + host flip —
    bit for bit, and the averaged probabilities match the oracle."""
    from PIL import Image

    from dfd import dropin
    from oracle import siglip_ref as R

    m, c, sd, hs = _bc("A")
    rng = np.random.default_rng(5)
    rows = []
    for i in range(7):
        arr = np.clip(rng.normal(128, 60, (40 + 3 * i, 50 + 2 * i, 3)), 0, 255).astype(np.uint8)
        Image.fromarray(arr).save(os.path.join(tmp_path, f"img{i}.png"))
        rows.append(f"img{i}.png,{i % 2}")
    rows.append("missing.png,1")   # rows without a file are dropped (:168-169)
    csv = os.path.join(tmp_path, "meta.csv")
    open(csv, "w").write("file_name,label\n" + "\n".join(rows) + "\n")
    tfs = dropin.create_tta_transforms(c.image_size, 2)
    assert [n for n, _ in tfs] == ["Original", "H-Flip"]
    y, p_avg, per, files = dropin.run_tta_inference(m, tmp_path, csv, tfs, batch_size=3, num_workers=0, device=torch.device(DEV))
    assert y.tolist() == [0, 1, 0, 1, 0, 1, 0] and files[3] == "img3.png" and len(per) == 2
    # the reference's way: one pass per transform, flip done by the host transform
    ref_passes = []
    for _, tf in tfs:
        ds = dropin.AIHumanDataset(tmp_path, csv, transform=tf)
        loader = torch.utils.data.DataLoader(ds, batch_size=3, shuffle=False)
        ref_passes.append(dropin.run_inference(m, loader, torch.device(DEV))[1])
    assert np.array_equal(per[0], ref_passes[0]) and np.array_equal(per[1], ref_passes[1])
    assert np.array_equal(p_avg, np.mean(ref_passes, axis=0))
    assert np.abs(per[0] - per[1]).max() > 1e-4      # the mirrored view really is a different input
    # oracle on the host-transformed tensors
    ds0 = dropin.AIHumanDataset(tmp_path, csv, transform=tfs[1][1])
    xf = torch.stack([ds0[i][0] for i in range(len(ds0))])
    pr = torch.sigmoid(R.classifier_head(hs, "A", R.siglip_vision_forward(sd, c, xf, "fp32")["pooler_output"], 0.0)).numpy()
    assert np.abs(per[1] - pr).max() < 1e-2      # 128-wide toy model, production engine mode (see test_binary_classifier_forward)
    # three transforms: the third (CLAHE) runs as an ordinary extra pass
    y3, p3, per3, _ = dropin.run_tta_inference(m, tmp_path, csv, dropin.create_tta_transforms(c.image_size, 3), 4, 0, torch.device(DEV))
    assert len(per3) == 3 and np.array_equal(per3[0], per[0]) and np.array_equal(per3[1], per[1])
    assert np.allclose(p3, np.mean(per3, axis=0))
    # Resize((S,S)) on the device too: the workers only decode (decode_only + ragged_collate), dfd_resize_u8 is bit-exact with PIL
    # and the patch kernel's ToTensor + Normalize lands on the same bf16 pixels as the host transform
    yd, pd_, perd, filesd = dropin.run_tta_inference(m, tmp_path, csv, tfs, batch_size=3, num_workers=0, device=torch.device(DEV),
                                                     device_resize=True)
    assert yd.tolist() == y.tolist() and filesd == files
    assert np.abs(perd[0] - per[0]).max() < 1e-3 and np.abs(perd[1] - per[1]).max() < 1e-3, (perd[0], per[0])
    ds_r = dropin.AIHumanDataset(tmp_path, csv, transform=dropin.decode_only)
    ld = torch.utils.data.DataLoader(ds_r, batch_size=3, shuffle=False, collate_fn=dropin.ragged_collate)
    assert np.abs(dropin.run_inference(m, ld, torch.device(DEV))[1] - per[0]).max() < 1e-3
    S_ = c.image_size
    for i in range(len(ds_r)):     # the resized pixels themselves, against the host transform's (before ToTensor)
        host = torch.round((dropin.AIHumanDataset(tmp_path, csv, transform=tfs[0][1])[i][0] * 0.5 + 0.5) * 255.0)
        dev = dropin.resize_on_device(m, [ds_r[i][0]])[0].cpu()
        assert dev.shape == (S_, S_, 3) and torch.equal(dev, host.permute(1, 2, 0).to(torch.uint8))


@pytest.mark.parametrize("fmt", ["u8", "f32"])
@pytest.mark.parametrize("S,P,Hin", [(64, 16, 64), (60, 14, 60), (60, 14, 37)])
def test_patchify_flip_equals_flipped_input(fmt, S, P, Hin):
    """DFD_FLIP_H: mirrored read of the source image == patchify of the host-flipped image, bit for bit, on the fast
    row kernel (u8, on-grid), the generic kernel (f32) and through the in-model bilinear resample (off-grid input)."""
    from dfd import ops
    from oracle import siglip_ref as R

    img = R.synthetic_images(3, Hin, seed=S + Hin)
    src = img if fmt == "u8" else R.preprocess_u8(img)
    flipped = torch.flip(src, dims=[2] if fmt == "u8" else [3]).contiguous()
    mode = ops.RESIZE_NONE if Hin == S else ops.RESIZE_BILINEAR
    a = ops.patchify(src.to(DEV), S, P, resize_mode=mode | ops.FLIP_H)
    b = ops.patchify(flipped.to(DEV), S, P, resize_mode=mode)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert not torch.equal(a, ops.patchify(src.to(DEV), S, P, resize_mode=mode))


def test_cifake_evaluate_vs_oracle():
    """cifake_binary_classifier.py:893-953 (BASELINE config 4): 32x32 images, bilinear 32 -> S inside the model, head H-D,
    BCE-with-logits, the reference's metric tuple — against the oracle flow on the same tensors."""
    from dfd import cifake, dropin
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd64"]
    sd = R.init_state_dict(c, 0)
    hd = R.init_head_d("small", c.hidden_size, 4)
    m = dropin.FastBinaryClassifier("small", DEV, arch="tiny-hd64", max_batch=16)
    ck = {"backbone.vision_model." + k: v for k, v in sd.items()}
    ck.update(hd)
    m.load_state_dict(ck)
    img = R.synthetic_images(22, 32, 8)
    labels = torch.tensor([0, 1] * 11)
    x = R.preprocess_u8(img)
    xr = R.resize_input(x, c.image_size, "bilinear")
    z_ref = R.classifier_head_d(hd, R.siglip_vision_forward(sd, c, xr, "fp32")["pooler_output"])
    p_ref = torch.sigmoid(z_ref).numpy()
    bs = 8
    for src in (x, img):   # float NCHW batches (the reference's loaders) and uint8 NHWC batches
        loader = [(src[i:i + bs], labels[i:i + bs]) for i in range(0, 22, bs)]
        loss, acc, bacc, prec, rec, f1, auc, mcc, cm, y, probs = cifake.evaluate(m, loader, torch.nn.BCEWithLogitsLoss(), torch.device(DEV))
        assert y.tolist() == labels.tolist() and probs.shape == (22,)
        assert np.abs(probs - p_ref).max() < 1e-2
        loss_ref = np.mean([float(torch.nn.functional.binary_cross_entropy_with_logits(z_ref[i:i + bs], labels[i:i + bs].float()))
                            for i in range(0, 22, bs)])
        assert abs(loss - loss_ref) < 1e-2
        sure = np.abs(p_ref - 0.5) > 2e-2                      # samples whose decision cannot flip within the tolerance
        assert ((probs > 0.5) == (p_ref > 0.5))[sure].all()
        assert cm.shape == (2, 2) and cm.sum() == 22 and 0.0 <= auc <= 1.0 and -1.0 <= mcc <= 1.0
        if sure.all():
            assert acc == float(((p_ref > 0.5) == labels.numpy()).mean())
    # TTA variant runs (random views: statistical check only — the mean stays near the base prediction)
    g = torch.Generator().manual_seed(0)
    z_tta = cifake.test_time_augmentation(m, img.to(DEV), n_tta=3, generator=g).cpu()
    assert z_tta.shape == (22,) and torch.isfinite(z_tta).all()
    sweep = cifake.throughput_sweep(m, batches=(16, 32), iters=1)
    assert set(sweep) == {16, 32} and all(v > 0 for v in sweep.values())


# ---------------------------------------------------------------------------------------------------------------------
# SURVEY §8 f.2: multicrop / rot-90 / patch-grid / video views produced on the device from one upload per image
# ---------------------------------------------------------------------------------------------------------------------
def _toy_pipeline(name="tiny-hd64", max_batch=32):
    from dfd import pipeline, scoring
    from oracle import siglip_ref as R
    from tests.conftest import SIGLIP_ARTEFACTS

    c = R.CONFIGS[name]
    sd, hs = R.init_state_dict(c, 0), R.init_head("B", c.hidden_size, 1)
    st = scoring.ScoringStack.from_dir(SIGLIP_ARTEFACTS, DEV)
    return pipeline.DetectionPipeline(name, sd, hs, st, device=0, max_batch=max_batch), c, sd, hs


def _pils(n, seed=3):
    from PIL import Image

    rng = np.random.default_rng(seed)
    return [Image.fromarray(np.clip(rng.normal(120, 50, (90 + 21 * i, 131 - 9 * i, 3)), 0, 255).astype(np.uint8)) for i in range(n)]


@pytest.mark.parametrize("clahe", [False, True])
def test_views_on_device_are_bit_exact_with_pil(clahe):
    """Every view (crop + PIL-exact resize for the model, crop + luma [+ CLAHE] + bicubic 256 for the frequency branch) built
    on the device from the resident original equals what the reference builds on the host with PIL / cv2, bit for bit."""
    from PIL import Image

    from dfd.scoring import pil_to_gray256

    pipe, c, _, _ = _toy_pipeline()
    S = c.image_size
    for pil in _pils(2):
        w, h = pil.size
        img = pipe._upload(pil)
        for maker in (pipe.multicrop_rects_v2, pipe.multicrop_rects_v3):
            rects, _ = maker(w, h)
            x, g = pipe.views_on_device(img, rects, clahe)
            torch.cuda.synchronize()
            assert x.shape == (len(rects), S, S, 3) and g.shape == (len(rects), 256, 256)
            for i, r in enumerate(rects):
                crop = pil.resize((S, S), Image.BICUBIC) if r == "bicubic" else pil.crop(r)
                ref_x = np.asarray(crop.resize((S, S), Image.BILINEAR))          # transforms.Resize((S,S)) on a PIL image
                assert np.array_equal(x[i].cpu().numpy(), ref_x), (r, "model input")
                assert np.array_equal(g[i].cpu().numpy(), pil_to_gray256(crop, clahe)), (r, "gray256")
        rot = pipe.rotate90_noexpand(img).cpu().numpy()
        assert np.array_equal(rot, np.asarray(pil.rotate(90, expand=False)))


def test_detect_core_device_equals_host_preprocessed_detect_core():
    """Same 6-view flow, views made on the device vs on the host (the path test_detect_core_multicrop_vs_oracle pins to the
    oracle): identical inputs reach the engine, so the results agree to fp32 rounding of the tiny weight sums."""
    pipe, _, _, _ = _toy_pipeline()
    pils = _pils(3)
    a = pipe.detect_core(pils, multicrop=True, clahe=False)
    b = pipe.detect_core_device(pils, views="v2", clahe=False)
    for ra, rb in zip(a, b):
        for k in ("z_sig", "z_freq", "z_scaled", "p_fake_raw", "p_fake_coral", "p_blend", "entropy"):
            assert abs(ra[k] - rb[k]) < 2e-6, (k, ra[k], rb[k])
        assert ra["risk_idx"] == rb["risk_idx"]
    one_a = pipe.detect_core(pils[:1], multicrop=False)
    one_b = pipe.detect_core_device(pils[:1], views=None)
    assert abs(one_a[0]["z_sig"] - one_b[0]["z_sig"]) < 2e-6 and abs(one_a[0]["z_freq"] - one_b[0]["z_freq"]) < 2e-6


def test_detect_core_v3_nine_crops_and_rot90_vs_oracle():
    """appv3.py:3214-3260 + :3315-3350: 9-crop weighted logits, 90-degree dual view (0.6 / 0.4 on probabilities, back to a
    logit), G1 fusion on probabilities, temperature, CORAL — restated with PIL + the oracle, vs one batched device call."""
    import json
    import math

    from safetensors.torch import load_file

    from dfd import dropin
    from oracle import scoring_ref as S
    from oracle import siglip_ref as R
    from tests.conftest import SIGLIP_ARTEFACTS

    pipe, c, sd, hs = _toy_pipeline()
    pils = _pils(2, seed=9)
    res = pipe.detect_core_device(pils, views="v3", rot90=True, clahe=False)
    fm, fu = load_file(f"{SIGLIP_ARTEFACTS}/freq_mlp.safetensors"), load_file(f"{SIGLIP_ARTEFACTS}/fusion_head.safetensors")
    cuts = S.coral_cut_logits(json.load(open(f"{SIGLIP_ARTEFACTS}/coral_cutpoints.json")))
    temp = json.load(open(f"{SIGLIP_ARTEFACTS}/coral_temp.json"))["temperature"]
    pre = dropin.make_preprocess(c.image_size, "bilinear")

    def z_of(views):
        x = torch.stack([pre(v) for v in views])
        return R.classifier_head(hs, "B", R.siglip_vision_forward(sd, c, x, "fp32")["pooler_output"], 1e-6).numpy()

    for pil, r in zip(pils, res):
        rects, w = pipe.multicrop_rects_v3(*pil.size)
        crops = [pil.crop(rc) for rc in rects]
        w = np.array(w, np.float32)
        z_sig = float((z_of(crops) * w).sum())
        z_rot = float(z_of([pil.rotate(90, expand=False)])[0])
        p = 0.6 / (1 + math.exp(-z_sig)) + 0.4 / (1 + math.exp(-z_rot))
        p = min(max(p, 1e-6), 1 - 1e-6)
        z_sig2 = math.log(p / (1 - p))
        assert abs(r["z_sig"] - z_sig2) < 3e-2, (r["z_sig"], z_sig2)      # toy 128-wide model, 10 bf16 forwards combined
        assert abs(r["visual_prob"] - p) < 1e-2
        # frequency branch + fusion + CORAL on the device's own z_sig: exact arithmetic of the reference flow
        host = pipe.detect_core([pil], multicrop=False)  # only to get the G1 parameters exercised the same way
        assert set(host[0]) == set(r)
        p_sig, p_freq = 1 / (1 + math.exp(-r["z_sig"])), 1 / (1 + math.exp(-r["z_freq"] / 1.25))
        z = float(fu["fc.weight"][0, 0]) * p_sig + float(fu["fc.weight"][0, 1]) * p_freq + float(fu["fc.bias"][0])
        d = S.detect_scores(np.array([z], np.float32), cuts, temp)
        assert abs(r["z_scaled"] - float(d["z_scaled"][0])) < 1e-4 and abs(r["p_blend"] - float(d["p_blend"][0])) < 1e-4
        tp = S.coral_transition_points(cuts)
        if np.abs(float(d["z_scaled"][0]) - tp).min() > 1e-3:
            assert r["risk_idx"] == int(d["risk_idx"][0])


def test_patch_grid_equals_per_cell_calls():
    """compute_patch_grid (app.py:1461-1485): all 16 cells in one batch == one single-view call per cell."""
    pipe, _, _, _ = _toy_pipeline()
    pil = _pils(1, seed=4)[0].resize((150, 97))
    grid, flat = pipe.patch_grid(pil, 4, 4)
    assert grid.shape == (4, 4) and len(flat) == 16
    rects = pipe.patch_grid_rects(150, 97, 4, 4)
    assert rects[3] == (111, 0, 150, 24) and rects[15] == (111, 72, 150, 97)      # last column / row take the remainder
    for i in (0, 3, 6, 15):
        cell = pipe.detect_core_device([pil.crop(rects[i])], views=None)[0]["p_fake_raw"]
        assert abs(cell - flat[i]) < 5e-6, (i, cell, flat[i])
    assert pipe.patch_grid(pil.resize((40, 80))) == (None, [])                     # below MIN_SIDE


def test_frame_features_vs_oracle():
    """hidf_video_classifier.py:299-320: frames -> encode_image -> L2 normalise -> mean over frames."""
    from oracle import siglip_ref as R

    pipe, c, sd, _ = _toy_pipeline()
    frames = R.synthetic_images(5, c.image_size, 12)
    f = pipe.frame_features(frames).cpu()
    ref = R.l2_normalize(R.siglip_vision_forward(sd, c, R.preprocess_u8(frames), "fp32")["pooler_output"])
    assert R.cosine_report(f, ref)["cos_min"] >= 0.999
    assert (f.norm(dim=-1) - 1).abs().max() < 1e-4
    assert R.cosine_report(f.mean(0, keepdim=True), ref.mean(0, keepdim=True))["cos_min"] >= 0.9995


@pytest.mark.parametrize("size", [280, 154])
def test_interpolate_pos_encoding_vs_hf(size):
    """HF `interpolate_pos_encoding=True` (HF:modeling_siglip.py:137-173; Siglip2sidafrozen.py:787 with the progressive
    resize of :975-987): inputs whose patch grid differs from the trained one (15x15 here -> 20x20 / 11x11) against the
    real transformers module in fp32, pooled output, last hidden state and every per-layer hidden state."""
    transformers = pytest.importorskip("transformers")
    from dfd import dropin
    from oracle import siglip_ref as R

    name = "small-hd72"
    c = R.CONFIGS[name]
    sd = R.init_state_dict(c, 0)
    hc = transformers.SiglipVisionConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                                         num_hidden_layers=c.num_hidden_layers, num_attention_heads=c.num_attention_heads,
                                         image_size=c.image_size, patch_size=c.patch_size)
    hf = transformers.SiglipVisionModel(hc).eval()
    hf.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
    x = R.preprocess_u8(R.synthetic_images(3, size, 5))
    with torch.no_grad():
        ref = hf(pixel_values=x, output_hidden_states=True, interpolate_pos_encoding=True)
    m = dropin.SiglipVisionModel.from_state_dict({"vision_model." + k: v for k, v in sd.items()}, DEV, max_batch=2,
                                                 num_heads=c.num_attention_heads)
    with pytest.raises(ValueError):
        m(pixel_values=x)                                   # like HF: a foreign grid needs the flag
    o = m(pixel_values=x, output_hidden_states=True, interpolate_pos_encoding=True)
    g = size // c.patch_size
    assert o.last_hidden_state.shape == (3, g * g, c.hidden_size) == tuple(ref.last_hidden_state.shape)
    rep = R.cosine_report(o.pooler_output.cpu(), ref.pooler_output)
    assert rep["cos_min"] >= 0.999 and rep["cos_centered_min"] >= 0.99 and rep["rel_l2"] <= 0.03, rep
    assert len(o.hidden_states) == len(ref.hidden_states) == c.num_hidden_layers + 1
    for a, b in zip(o.hidden_states, ref.hidden_states):
        r = R.cosine_report(a.cpu().reshape(-1, c.hidden_size), b.reshape(-1, c.hidden_size))
        assert r["cos_min"] >= 0.998 and r["rel_l2"] <= 0.03, r
    # the position table itself: bit-equal to HF's interpolation
    emb = hf.vision_model.embeddings
    want = emb.interpolate_pos_encoding(torch.zeros(1, g * g, c.hidden_size), size, size)[0]
    got = dropin.interpolated_position_table(sd["embeddings.position_embedding.weight"], g)
    assert torch.equal(got, want)
    # native-size calls keep using the native engine
    x0 = R.preprocess_u8(R.synthetic_images(2, c.image_size, 6))
    o0 = m(pixel_values=x0, interpolate_pos_encoding=True)
    with torch.no_grad():
        r0 = hf(pixel_values=x0, interpolate_pos_encoding=True)
    assert R.cosine_report(o0.pooler_output.cpu(), r0.pooler_output)["cos_min"] >= 0.999

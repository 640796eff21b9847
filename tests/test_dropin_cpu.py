"""CPU tests of the drop-in boundary (SURVEY.md §8b): the reference's OWN classes, extracted from its source text and
exec'd with the dfd `open_clip` stand-in installed, must register the dfd vision tower as a submodule and deliver the
checkpoint's `backbone.*` tensors into it through their own load paths (inference_ai_human_images.py:841-857,
train_fusion_head_only.py:111-124).  No forward runs here (no GPU: the tower is a parameter skeleton and its forward
raises); the numerics of the same flow are checked on the GPU in tests/test_dropin_gpu.py.

The reference's source is not part of this repository: the tests that exec it read a checkout named by DFD_REFERENCE_DIR
and skip without one.  They also pin tests/reference_style.py, the restatement of the same classes that the test_restated_*
tests here and the GPU tests drive on every machine, to the originals (same parameters, same loaded tensors).
"""
import ast
import os
import sys
import types
import warnings

import pytest
import torch
import torch.nn as nn

from tests.reference_style import load_siglip_from_best, reference_style_classifier

REF = os.environ.get("DFD_REFERENCE_DIR", "")
needs_ref = pytest.mark.skipif(not os.path.isdir(REF), reason="DFD_REFERENCE_DIR does not name a checkout of the reference")


def _extract(path, names):
    """Source text of the named top-level classes / functions of a reference file."""
    src = open(path, encoding="utf-8").read()
    tree = ast.parse(src)
    out = []
    for node in tree.body:
        if isinstance(node, (ast.ClassDef, ast.FunctionDef)) and node.name in names:
            out.append(ast.get_source_segment(src, node))
    assert len(out) == len(names), f"{path}: found {len(out)} of {names}"
    return "\n\n".join(out)


@pytest.fixture()
def shims(monkeypatch):
    from dfd import dropin
    from dfd.engine import ARCHS

    # the reference hard-codes ViT-B/L-16-SigLIP-384; map those names to toy trunks so the CPU test stays small
    monkeypatch.setitem(dropin.ARCHS, "ViT-B-16-SigLIP-384", ARCHS["tiny-hd64"])
    monkeypatch.setitem(dropin.ARCHS, "ViT-L-16-SigLIP-384", ARCHS["tiny-hd72"])
    for m in ("open_clip", "pywt"):
        monkeypatch.delitem(sys.modules, m, raising=False)
    dropin.install_import_shims()
    yield dropin
    for m in ("open_clip", "pywt"):
        sys.modules.pop(m, None)


def _checkpoint_like(model, seed):
    """A checkpoint as open_clip + the reference's trainers write it: every tensor of the model's own state dict (fresh
    values), plus the text tower and the scalar logit parameters of the full open_clip model."""
    g = torch.Generator().manual_seed(seed)
    ck = {k: torch.randn(v.shape, generator=g) for k, v in model.state_dict().items()}
    ck["backbone.logit_scale"] = torch.tensor(2.3)
    ck["backbone.logit_bias"] = torch.tensor(-10.0)
    ck["backbone.text.transformer.resblocks.0.ln_1.weight"] = torch.ones(8)
    ck["backbone.text.token_embedding.weight"] = torch.zeros(4, 8)
    return ck


def _param_shapes(model):
    return {k: tuple(v.shape) for k, v in model.state_dict().items()}


def _restated(kind, shims):
    name, img_size = ("ViT-B-16-SigLIP-384", 64) if kind == "A" else ("ViT-L-16-SigLIP-384", 60)
    return reference_style_classifier(kind, name, shims.ARCHS[name].hidden_size, img_size)


def _check_inference_classifier_strict_load(make):
    """The load path of inference_ai_human_images.py (:841-857) on the model `make()` builds; returns the model."""
    with pytest.warns(UserWarning, match="random"):   # pretrained='webli' cannot be fetched: said loudly, not silently
        model = make()
    assert isinstance(model.backbone, nn.Module) and "backbone" in dict(model.named_children())
    names = [k for k, _ in model.named_parameters()]
    assert "backbone.visual.trunk.blocks.1.attn.qkv.weight" in names            # timm names (simple_classifier.py:491)
    assert "backbone.visual.trunk.attn_pool.latent" in names and "backbone.visual.trunk.pos_embed" in names
    assert model.backbone.weights_source == "random"
    ck = _checkpoint_like(model, 1)
    model.load_state_dict(ck, strict=True)     # the reference's first attempt; must not need the non-strict fallback
    assert model.backbone.weights_source == "checkpoint"
    for k, v in model.state_dict().items():
        assert torch.equal(v, ck[k]), k
    # the fallback path unpacks torch's NamedTuple (:850)
    missing_keys, unexpected_keys = model.load_state_dict({k: v for k, v in ck.items() if "classifier" in k}, strict=False)
    assert len(unexpected_keys) == 0 and all(k.startswith("backbone.") for k in missing_keys) and missing_keys
    # a head-only checkpoint leaves the backbone untouched and the tower knows it still has what it had
    assert model.backbone.weights_source == "checkpoint"
    with pytest.raises(RuntimeError, match="CUDA"):
        model(torch.zeros(1, 3, 64, 64))       # no CPU fallback: the forward fails loudly
    return model


@needs_ref
def test_reference_inference_classifier_strict_load_reaches_the_backbone(shims):
    """inference_ai_human_images.py: `BinaryClassifier(nn.Module)` + its strict load (:841-846)."""
    import open_clip  # the stand-in

    ns = {"torch": torch, "nn": nn, "open_clip": open_clip, "print": lambda *a, **k: None}
    exec(_extract(os.path.join(REF, "inference_ai_human_images.py"), ["BinaryClassifier"]), ns)
    model = _check_inference_classifier_strict_load(lambda: ns["BinaryClassifier"](model_size="small", device="cpu").to("cpu"))
    # the restatement the other tests drive declares the same submodules and parameters
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        restated = _restated("A", shims)("cpu")
    assert [n for n, _ in restated.named_children()] == [n for n, _ in model.named_children()]
    assert _param_shapes(restated) == _param_shapes(model)


def test_restated_inference_classifier_strict_load_reaches_the_backbone(shims):
    """The same load path on tests/reference_style.py's restatement of that class (no reference checkout needed)."""
    _check_inference_classifier_strict_load(lambda: _restated("A", shims)("cpu").to("cpu"))


def _check_fusion_trainer_loader(classifier, load_from_best, tmp_path):
    """`load_siglip_from_best` of train_fusion_head_only.py (:111-124) on a synthetic `best_model` checkpoint of `classifier`:
    every trunk tensor arrives.  Returns (probe, loaded model, checkpoint path)."""
    from safetensors.torch import save_file

    with pytest.warns(UserWarning):
        probe = classifier("cpu")
    ck = _checkpoint_like(probe, 2)
    path = os.path.join(tmp_path, "best_model.safetensors")
    save_file({k: v.contiguous() for k, v in ck.items()}, path)
    with pytest.warns(UserWarning):
        model = load_from_best(path)
    assert model.backbone.weights_source == "checkpoint"
    sd = model.state_dict()
    n_backbone = 0
    for k, v in sd.items():
        assert torch.equal(v, ck[k]), k
        n_backbone += k.startswith("backbone.visual.trunk.")
    assert n_backbone == 12 * probe.backbone.arch.num_hidden_layers + 18   # every trunk tensor went through the filter
    return probe, model, path


@needs_ref
def test_reference_fusion_trainer_loader_reaches_the_backbone(shims, tmp_path):
    """train_fusion_head_only.py: `BinaryClassifier`, `_filter_state_for_model`, `load_siglip_from_best` (:78-124)."""
    import open_clip
    from safetensors.torch import load_file

    D = shims.ARCHS["ViT-L-16-SigLIP-384"].hidden_size
    ns = {"torch": torch, "nn": nn, "open_clip": open_clip, "load_file": load_file, "SIGLIP_DIM": D, "IMG_SIZE": 60,
          "DEVICE": "cpu", "print": lambda *a, **k: None}
    exec(_extract(os.path.join(REF, "train_fusion_head_only.py"),
                  ["BinaryClassifier", "_filter_state_for_model", "load_siglip_from_best"]), ns)
    probe, model, path = _check_fusion_trainer_loader(ns["BinaryClassifier"], ns["load_siglip_from_best"], tmp_path)
    # the restatement declares the same submodules and parameters, and its loader delivers the same tensors
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        restated = _restated("B", shims)
        assert [n for n, _ in restated("cpu").named_children()] == [n for n, _ in probe.named_children()]
        assert _param_shapes(restated("cpu")) == _param_shapes(probe)
        mine = load_siglip_from_best(restated, path)
    theirs = model.state_dict()
    assert all(torch.equal(v, theirs[k]) for k, v in mine.state_dict().items())


def test_restated_fusion_trainer_loader_reaches_the_backbone(shims, tmp_path):
    """The same loader on tests/reference_style.py's restatement (no reference checkout needed)."""
    restated = _restated("B", shims)
    _check_fusion_trainer_loader(restated, lambda path: load_siglip_from_best(restated, path), tmp_path)


def test_tower_accepts_hf_layout_and_round_trips_timm_names():
    from dfd import dropin
    from dfd.engine import ARCHS
    from oracle import siglip_ref as R

    c = R.CONFIGS["tiny-hd72"]
    sd = R.init_state_dict(c, 0)
    tower = dropin.VisionTower(ARCHS["tiny-hd72"], "cpu", state_dict=sd)
    assert tower.weights_source == "state_dict"
    own = tower.state_dict()
    D = c.hidden_size
    assert torch.equal(own["visual.trunk.blocks.1.attn.qkv.weight"],
                       torch.cat([sd[f"encoder.layers.1.self_attn.{x}_proj.weight"] for x in "qkv"], 0))
    assert torch.equal(own["visual.trunk.attn_pool.kv.bias"], sd["head.attention.in_proj_bias"][D:])
    assert own["visual.trunk.pos_embed"].shape == (1, c.image_size // c.patch_size * (c.image_size // c.patch_size), D)
    # HF-layout checkpoint through nn.Module.load_state_dict (strict) on a fresh tower
    with pytest.warns(UserWarning):
        t2 = dropin.create_model_and_transforms("tiny-hd72", pretrained="webli", device="cpu")[0]
    r = t2.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
    assert not r.missing_keys and not r.unexpected_keys and t2.weights_source == "checkpoint"
    for k, v in t2.state_dict().items():
        assert torch.equal(v, own[k]), k
    # and the engine-side mapping is the inverse: timm names -> canonical names
    from dfd.engine import canonicalize_state_dict

    canon = canonicalize_state_dict(own)
    for k, v in sd.items():
        if "self_attn.q_proj" in k or "self_attn.k_proj" in k or "self_attn.v_proj" in k:
            continue
        assert torch.equal(canon[k].reshape(v.shape), v), k


def test_unexpected_backbone_keys_are_reported():
    from dfd import dropin
    from dfd.engine import ARCHS

    tower = dropin.VisionTower(ARCHS["tiny-hd64"], "cpu")
    sd = dict(tower.state_dict())
    sd["visual.trunk.blocks.0.attn.q_norm.weight"] = torch.ones(4)
    sd["bogus.weight"] = torch.ones(1)
    with pytest.raises(RuntimeError, match="Unexpected"):
        tower.load_state_dict(sd, strict=True)
    r = tower.load_state_dict(sd, strict=False)
    assert set(r.unexpected_keys) == {"visual.trunk.blocks.0.attn.q_norm.weight", "bogus.weight"}

"""The reference's two `BinaryClassifier` classes and its checkpoint loader, restated the way the reference declares them
(same submodule names, same forward, same load path), for the tests that run without a checkout of the reference:
tests/test_dropin_gpu.py drives them on the GPU, tests/test_dropin_cpu.py on the CPU.  Where DFD_REFERENCE_DIR names a
checkout, tests/test_dropin_cpu.py also checks them against the reference's own source: same parameters, same loaded tensors."""
import torch
import torch.nn as nn


def reference_style_classifier(kind, arch_name, dim, img_size):
    """kind 'A': inference_ai_human_images.py:111-152; kind 'B': train_fusion_head_only.py:78-109."""
    import open_clip  # the dfd stand-in (install_import_shims)

    class BinaryClassifierA(nn.Module):
        def __init__(self, device):
            super().__init__()
            self.resolution = img_size
            self.backbone, _, self.preprocess = open_clip.create_model_and_transforms(arch_name, pretrained="webli", device=device)
            self.classifier = nn.Sequential(nn.LayerNorm(dim), nn.Dropout(0.3), nn.Linear(dim, dim // 2), nn.GELU(),
                                            nn.Dropout(0.2), nn.Linear(dim // 2, 1))

        def forward(self, x):
            features = self.backbone.encode_image(x)
            features = features / features.norm(dim=-1, keepdim=True)
            return self.classifier(features).squeeze(-1)

    class BinaryClassifierB(nn.Module):
        def __init__(self, device):
            super().__init__()
            self.backbone, _, _ = open_clip.create_model_and_transforms(arch_name, pretrained="webli", device=device)
            self.se = nn.Sequential(nn.Linear(dim, dim // 16), nn.ReLU(), nn.Linear(dim // 16, dim), nn.Sigmoid())
            self.classifier = nn.Sequential(nn.LayerNorm(dim), nn.Dropout(0.3), nn.Linear(dim, dim // 2), nn.GELU(),
                                            nn.Dropout(0.2), nn.Linear(dim // 2, dim // 4), nn.GELU(), nn.Linear(dim // 4, 1))

        def forward(self, x):
            with torch.no_grad():
                if x.shape[-1] != img_size:
                    x = nn.functional.interpolate(x, size=(img_size, img_size))
                f = self.backbone.encode_image(x)
                f = f / (f.norm(dim=-1, keepdim=True) + 1e-6)
            return self.classifier(f * self.se(f)).squeeze(-1)

    return BinaryClassifierA if kind == "A" else BinaryClassifierB


def load_siglip_from_best(classifier, path, device="cpu"):
    """train_fusion_head_only.py:111-124: `BinaryClassifier(DEVICE)`, `load_file`, then a non-strict load of the tensors whose
    names and shapes the model has (`_filter_state_for_model`)."""
    from safetensors.torch import load_file

    model = classifier(device)
    own = model.state_dict()
    state = {k: v for k, v in load_file(path).items() if k in own and tuple(own[k].shape) == tuple(v.shape)}
    model.load_state_dict(state, strict=False)
    return model

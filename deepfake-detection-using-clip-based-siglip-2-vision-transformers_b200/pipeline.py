"""DetectionPipeline — the batched form of the reference's `detect_core` (deepfake-detector-v2/app.py:1329-1412)
and of the extraction loops of train_fusion_head_only.py:329-347:

    images (u8 NHWC) ──SigLIP engine──> pooled ──classifier head──> z_sig ┐
       └─ gray256 kernels (luma, CLAHE, bicubic 256²) ─ freq feature kernels ─> 24-d features ─┴─ score epilogue ──> z, CORAL
    (gray256 may also be handed in, e.g. when the caller's images are not at the model resolution)

One call = (7·L + 13) backbone launches + head + 2 freq kernels + 1 score-epilogue kernel, all enqueue-only on the
current stream; `detect()` adds the pinned H2D copies and one D2H read of the packed scores, which is what the
reference loops do per batch (inference_ai_human_images.py:274,296).
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from . import ops
from .engine import ARCHS, SiglipEngine, VisionArch
from .scoring import EPS_TRAINER, FreqFeatureExtractor, ScoringStack

PACKED_FIELDS = ("z_sig", "z_freq", "z", "z_scaled", "p_raw", "p_coral", "entropy", "p_blend", "risk_idx",
                 "risk_p0", "risk_p1", "risk_p2", "risk_p3", "risk_p4")


def head_params_from_state(sd: Dict[str, torch.Tensor], dim: int, device) -> "ops.HeadParams":
    """`BinaryClassifier` / `FastBinaryClassifier` heads (SURVEY.md §8 a7), recognised by their key names:
      H-A  classifier.{0,2,5}                 inference_ai_human_images.py:131-138 (no eps on the L2 norm)
      H-B  se.{0,2} + classifier.{0,2,5,7}    train_fusion_head_only.py:84-99 (norm + 1e-6)
      H-D  layer_norm + [attention.*] + classifier.{0,3[,6]} or {1}   cifake_binary_classifier.py:643-684,728-749
           (attention over ONE token is exactly proj(v(x)): softmax of a single score is 1)"""
    G, N = ops.ACT_GELU, ops.ACT_NONE
    if "layer_norm.weight" in sd:  # H-D
        layers = []
        if "attention.qkv.weight" in sd:        # LightweightAttention: rows [2D,3D) of the fused qkv are v
            layers += [(sd["attention.qkv.weight"][2 * dim:], sd["attention.qkv.bias"][2 * dim:], N),
                       (sd["attention.proj.weight"], sd["attention.proj.bias"], N)]
        elif "attention.in_proj_weight" in sd:  # nn.MultiheadAttention
            layers += [(sd["attention.in_proj_weight"][2 * dim:], sd["attention.in_proj_bias"][2 * dim:], N),
                       (sd["attention.out_proj.weight"], sd["attention.out_proj.bias"], N)]
        idx = sorted(int(k.split(".")[1]) for k in sd if k.startswith("classifier.") and k.endswith(".weight"))
        for n, i in enumerate(idx):
            layers.append((sd[f"classifier.{i}.weight"], sd[f"classifier.{i}.bias"], G if n + 1 < len(idx) else N))
        return ops.HeadParams(1, dim, 0.0, device, ln=(sd["layer_norm.weight"], sd["layer_norm.bias"]), layers=layers)
    ln = (sd["classifier.0.weight"], sd["classifier.0.bias"])
    if "se.0.weight" in sd:
        se = (sd["se.0.weight"], sd["se.0.bias"], sd["se.2.weight"], sd["se.2.bias"])
        layers = [(sd["classifier.2.weight"], sd["classifier.2.bias"], G), (sd["classifier.5.weight"], sd["classifier.5.bias"], G),
                  (sd["classifier.7.weight"], sd["classifier.7.bias"], N)]
        return ops.HeadParams(2, dim, 1e-6, device, ln=ln, se=se, layers=layers)
    layers = [(sd["classifier.2.weight"], sd["classifier.2.bias"], G), (sd["classifier.5.weight"], sd["classifier.5.bias"], N)]
    return ops.HeadParams(1, dim, 0.0, device, ln=ln, layers=layers)


def _on_own_device(fn):
    """Run a pipeline method with the pipeline's GPU as the current device (its kernels are launched on the current device's
    stream), whatever device the caller has selected."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)

    return wrapped


class DetectionPipeline:
    def __init__(self, arch: VisionArch | str, backbone_state: Dict[str, torch.Tensor],
                 head_state: Dict[str, torch.Tensor], scoring: ScoringStack, device: int = 0, max_batch: int = 64,
                 freq_eps: float = EPS_TRAINER, freq_zscore: Optional[bool] = None, fuse_ln: bool = True,
                 graphs: bool = False, precise_residual: bool = False):
        self.arch = ARCHS[arch] if isinstance(arch, str) else arch
        self.device = torch.device("cuda", device)
        self.engine = SiglipEngine(self.arch, device, max_batch, fuse_ln=fuse_ln, graphs=graphs,
                                   precise_residual=precise_residual).load_state_dict(backbone_state)
        self.head = head_params_from_state(head_state, self.arch.hidden_size, self.device)
        self.scoring = scoring
        # G1 heads were trained on z-scored vectors (app.py:840-846), G2 on raw ones + learned normaliser
        zs = (scoring.gen == 1) if freq_zscore is None else freq_zscore
        self.freq = FreqFeatureExtractor(self.device, eps=freq_eps, zscore=zs)
        self._pin: Dict[str, torch.Tensor] = {}
        self._gray_scratch: Optional[torch.Tensor] = None
        self._stage_ev = None    # measurement aid (bench.py): CUDA events around the non-backbone stages

    # ---- measurement aid: per-stage CUDA-event timing of the kernels outside the engine --------------------------------
    def profile_stages(self, enable: bool = True) -> None:
        self._stage_ev = [] if enable else None

    def profile_stages_read(self) -> Dict[str, tuple]:
        """{'head' | 'gray256' | 'freq' | 'score': (ms, calls)} since profiling was switched on; clears the record."""
        out: Dict[str, list] = {}
        if self._stage_ev:
            self._stage_ev[-1][2].synchronize()
            for name, a, b in self._stage_ev:
                acc = out.setdefault(name, [0.0, 0])
                acc[0] += a.elapsed_time(b)
                acc[1] += 1
            self._stage_ev = []
        return {k: (v[0], v[1]) for k, v in out.items()}

    def _stage(self, name, fn):
        if self._stage_ev is None:
            return fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        self._stage_ev.append((name, a, b))
        return r

    # ---- device-resident path ---------------------------------------------------------------------
    @_on_own_device
    def detect_device(self, images: torch.Tensor, gray256: Optional[torch.Tensor] = None, resize_mode: int = 0,
                      clahe: bool = True, pil_resize: Optional[str] = None) -> Dict[str, torch.Tensor]:
        """images: u8 NHWC on the device.  gray256 None = derive it from the same (original-size) pixels on the device
        (train_fusion_head_only.py:142-148 with clahe=True; app.py:736-749 with DETECT_USE_CLAHE for clahe).
        pil_resize "bilinear" / "bicubic": images of another size first go through the PIL-exact `Resize((S,S))` of the
        reference's transforms (inference_ai_human_images.py:200-204) instead of the in-model resize (resize_mode)."""
        S = self.arch.image_size
        model_in = images
        if pil_resize is not None and tuple(images.shape[1:3]) != (S, S):
            model_in = ops.resize_u8(images, S, S, pil_resize)
        pooled, _ = self.engine(model_in, resize_mode=resize_mode)
        _, z_sig, _ = self._stage("head", lambda: ops.head_fwd(self.head, pooled))
        if gray256 is None:
            need = ops._lib.load().dfd_gray256_scratch_bytes(*images.shape[:3])
            if self._gray_scratch is None or self._gray_scratch.numel() < need:
                self._gray_scratch = torch.empty((need,), dtype=torch.uint8, device=self.device)
            gray256 = self._stage("gray256", lambda: ops.gray256_from_rgb(images, clahe, scratch=self._gray_scratch))
        feats = self._stage("freq", lambda: self.freq.from_gray(gray256))
        out = self._stage("score", lambda: self.scoring(z_sig, feats=feats))
        out["pooled"] = pooled
        return out

    @_on_own_device
    def explain(self, images_u8: torch.Tensor, resize_mode: int = 0, alpha: float = 0.5) -> Dict[str, torch.Tensor]:
        """Where the backbone looks: attention rollout (Abnar & Zuidema 2020) seeded by the MAP pooling probe, the query
        that forms the pooled embedding.  images_u8: u8 NHWC on the device.  Returns {"relevance" [B,G,G] (sums to 1 per
        image), "heatmap" [B,S,S] (bilinear upsample of G²·relevance: 1.0 = a uniform share, above 1 = more than its
        share), "z_sig" [B] (the classifier logit of the same forward)}.  The maps are not normalised; to display one,
        scale it to [0, 1] per image (or clip at a fixed multiple of the uniform share) and overlay it on the image.
        Runs in chunks of at most max_batch images; the head-mean probabilities take L·N²·4 bytes per image."""
        a, eng = self.arch, self.engine
        G, S = a.grid, a.image_size
        rel, heat, z = [], [], []
        for i in range(0, images_u8.shape[0], eng.max_batch):
            pooled, attn, map_p = eng.forward_attentions(images_u8[i:i + eng.max_batch], resize_mode)
            r, h = ops.attention_rollout(attn, map_p, alpha, S)
            del attn
            rel.append(r.view(-1, G, G))
            heat.append(h)
            z.append(ops.head_fwd(self.head, pooled)[1])
        return {"relevance": torch.cat(rel), "heatmap": torch.cat(heat), "z_sig": torch.cat(z)}

    @staticmethod
    def pack(out: Dict[str, torch.Tensor]) -> torch.Tensor:
        """[B, 14] fp32 score records (PACKED_FIELDS) — the unit that is all-gathered across ranks."""
        cols = [out[k].float() for k in PACKED_FIELDS[:8]] + [out["risk_idx"].float()]
        return torch.cat([torch.stack(cols, 1), out["risk_probs"]], 1)

    # ---- detect_core: multicrop, one batched call (deepfake-detector-v2/app.py:1329-1412, 1418-1430) ---------------
    MULTICROP_WEIGHTS = (0.4, 0.4, 0.05, 0.05, 0.05, 0.05)

    def make_multicrops(self, pil):
        """The reference's 6 views: full image, bicubic S x S resize, four quadrants; weights .4/.4/.05x4."""
        from PIL import Image

        S = self.arch.image_size
        w, h = pil.size
        w2, h2 = max(1, w // 2), max(1, h // 2)
        return [pil, pil.resize((S, S), Image.BICUBIC), pil.crop((0, 0, w2, h2)), pil.crop((w2, 0, w, h2)),
                pil.crop((0, h2, w2, h)), pil.crop((w2, h2, w, h))]

    @torch.no_grad()
    @_on_own_device
    def detect_core(self, pils, multicrop: bool = True, clahe: bool = False, preprocess=None, freq_temp: float = 1.25):
        """Batched `detect_core`: every crop of every image goes through ONE backbone / feature batch, crop logits
        are combined with the reference's weights (on logits, app.py:1346-1347), then one score epilogue per image.
        Returns a list of dicts with the reference's keys."""
        import numpy as np

        from .dropin import make_preprocess
        from .scoring import pil_to_gray256

        pre = preprocess or make_preprocess(self.arch.image_size, "bilinear")
        views, wts = [], []
        for pil in pils:
            pil = pil.convert("RGB")
            cs = self.make_multicrops(pil) if multicrop else [pil]
            views += cs
            wts.append(list(self.MULTICROP_WEIGHTS) if multicrop else [1.0])
        nv = len(wts[0])
        x = torch.stack([pre(v) for v in views]).to(self.device, non_blocking=True)
        gray = torch.from_numpy(np.stack([pil_to_gray256(v, clahe) for v in views])).to(self.device, non_blocking=True)
        pooled, _ = self.engine(x)
        z_sig = ops.head_fwd(self.head, pooled)[1]
        z_freq = self.scoring(torch.zeros_like(z_sig), feats=self.freq.from_gray(gray))["z_freq"]
        w = torch.tensor(wts, dtype=torch.float32, device=self.device)
        zs = (z_sig.view(-1, nv) * w).sum(1).contiguous()
        zf = (z_freq.view(-1, nv) * w).sum(1).contiguous()
        out = self.scoring(zs, z_freq=zf)
        host = {k: v.cpu().numpy() for k, v in out.items()}
        res = []
        for i in range(len(pils)):
            zsi, zfi = float(host["z_sig"][i]), float(host["z_freq"][i])
            res.append({"z_sig": zsi, "z_freq": zfi, "z_scaled": float(host["z_scaled"][i]),
                        "p_fake_raw": float(host["p_raw"][i]), "p_fake_coral": float(host["p_coral"][i]),
                        "p_blend": float(host["p_blend"][i]), "visual_prob": 1.0 / (1.0 + np.exp(-zsi)),
                        "freq_prob": 1.0 / (1.0 + np.exp(-zfi / freq_temp)), "p_or": None, "p_moe": None,
                        "risk_idx": int(host["risk_idx"][i]), "risk_probs": torch.from_numpy(host["risk_probs"][i].copy()),
                        "entropy": float(host["entropy"][i])})
        return res

    # ---- streaming host-buffer path: the public throughput API ---------------------------------------------------------
    @_on_own_device
    def detect_many(self, batches, resize_mode: int = 0, clahe: bool = True, pil_resize: Optional[str] = None,
                    in_flight: int = 2, on_result=None):
        """Host u8 NHWC batches (an iterable; pinned tensors copy asynchronously) -> list of numpy [B_i,14] score records,
        in order.  The upload of batch k+1 and the download of batch k's records run on a copy stream under batch k's
        kernels (`in_flight` device input slabs, one pinned record buffer per batch in flight), so PCIe time leaves the
        critical path; `detect()` is the one-batch, fully synchronous form.  `on_result(k, records)` is called as each
        batch's records arrive (the per-batch `all_probs.extend(...)` point of the reference loops)."""
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(dev)
        cs = self._copy_stream
        slabs, free_ev, pend, out = [], [], [], []
        it = iter(batches)

        def upload(k, host):
            i = k % in_flight
            if len(slabs) <= i:
                slabs.append(None)
                free_ev.append(None)
            if slabs[i] is None or slabs[i].shape != host.shape:
                slabs[i] = torch.empty(host.shape, dtype=torch.uint8, device=dev)
            with torch.cuda.stream(cs):
                if free_ev[i] is not None:
                    cs.wait_event(free_ev[i])          # the kernels that read this slab (batch k - in_flight) are done
                slabs[i].copy_(host, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
            return slabs[i], ev

        def drain(limit):
            while len(pend) > limit:
                k, rec_host, ev = pend.pop(0)
                ev.synchronize()
                r = rec_host.numpy().copy()
                out.append(r)
                if on_result is not None:
                    on_result(k, r)

        nxt = next(it, None)
        k = 0
        staged = upload(0, nxt) if nxt is not None else None
        while staged is not None:
            img, up_ev = staged
            nxt = next(it, None)
            staged = upload(k + 1, nxt) if nxt is not None else None   # overlaps with the kernels enqueued below
            main.wait_event(up_ev)
            packed = self.pack(self.detect_device(img, None, resize_mode, clahe, pil_resize))
            done = torch.cuda.Event()
            done.record(main)
            free_ev[k % in_flight] = done
            rec_host = torch.empty(packed.shape, dtype=torch.float32).pin_memory()
            with torch.cuda.stream(cs):
                cs.wait_event(done)
                rec_host.copy_(packed, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
            packed.record_stream(cs)
            pend.append((k, rec_host, ev))
            drain(in_flight - 1)     # keeps the host at most `in_flight` batches ahead of the device
            k += 1
        drain(0)
        return out

    # ---- views produced ON THE DEVICE from one upload per image (SURVEY.md §8 f.2) ---------------------------------
    # The reference preprocesses every crop on the host (PIL resize + ToTensor per crop, PIL/cv2 gray256 per crop) and
    # runs ~50 batch-1 forwards per upload.  Here the original pixels cross PCIe once; every view is a rectangle of the
    # resident image that goes through dfd_resize_u8 (bit-exact PIL `Resize`) and dfd_gray256 (bit-exact luma / CLAHE /
    # bicubic 256x256), and all views of all images run as ONE engine batch.
    @staticmethod
    def multicrop_rects_v2(w: int, h: int):
        """deepfake-detector-v2/app.py:1418-1430: full image, bicubic S x S resize of it, four quadrants."""
        w2, h2 = max(1, w // 2), max(1, h // 2)
        rects = [(0, 0, w, h), "bicubic", (0, 0, w2, h2), (w2, 0, w, h2), (0, h2, w2, h), (w2, h2, w, h)]
        return rects, [0.4, 0.4, 0.05, 0.05, 0.05, 0.05]

    @staticmethod
    def multicrop_rects_v3(w: int, h: int):
        """appv3.py:3315-3350: centre (50 %), left / right / top / bottom halves, four quadrants; tiny images fall back to
        the bicubic S x S resize alone."""
        if w < 4 or h < 4:
            return ["bicubic"], [1.0]
        mw, mh = w // 2, h // 2
        cw, ch = max(1, w // 2), max(1, h // 2)
        cx0, cy0 = max(0, (w - cw) // 2), max(0, (h - ch) // 2)
        rects = [(cx0, cy0, cx0 + cw, cy0 + ch), (0, 0, mw, h), (w - mw, 0, w, h), (0, 0, w, mh), (0, h - mh, w, h),
                 (0, 0, mw, mh), (w - mw, 0, w, mh), (0, h - mh, mw, h), (w - mw, h - mh, w, h)]
        return rects, [0.20] + [0.10] * 8

    @staticmethod
    def patch_grid_rects(w: int, h: int, rows: int = 4, cols: int = 4, min_side: int = 64):
        """deepfake-detector-v2/app.py:1461-1485: rows x cols cells (last row / column take the remainder); None for
        images below MIN_SIDE, empty cells are None."""
        if w < min_side or h < min_side:
            return None
        pw, ph = max(8, w // cols), max(8, h // rows)
        out = []
        for r in range(rows):
            for c in range(cols):
                x0, y0 = c * pw, r * ph
                x1 = w if c == cols - 1 else min(w, x0 + pw)
                y1 = h if r == rows - 1 else min(h, y0 + ph)
                out.append((x0, y0, x1, y1) if (x1 > x0 and y1 > y0) else None)
        return out

    @staticmethod
    def rotate90_noexpand(img: torch.Tensor) -> torch.Tensor:
        """PIL `Image.rotate(90, expand=False)` (appv3.py:3241) of a u8 [H,W,3] device image: counter-clockwise quarter turn
        about the centre on the SAME canvas; for non-square images the parts that leave the canvas are dropped and the
        uncovered area is black.  Pure index arithmetic (PIL's affine NEAREST path with an exact 0 / 1 matrix)."""
        H, W = img.shape[:2]
        if H == W:
            return torch.rot90(img, 1, (0, 1)).contiguous()      # PIL special-cases squares: transpose(ROTATE_90)
        dev = img.device
        # PIL: matrix = [cos, sin, c; -sin, cos, f] with angle = -90 deg, cos / sin rounded to 15 digits -> [0, -1; 1, 0],
        # c, f = matrix applied to minus the centre, plus the centre; output pixel centre (x + .5, y + .5) maps to the input
        # point (xin, yin); NEAREST takes floor, points outside the canvas give the fill colour 0.
        cx, cy = W / 2.0, H / 2.0
        ys, xs = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float64) + 0.5,
                                torch.arange(W, device=dev, dtype=torch.float64) + 0.5, indexing="ij")
        a, b, d, e = 0.0, -1.0, 1.0, 0.0
        c = a * -cx + b * -cy + cx
        f = d * -cx + e * -cy + cy
        xin = a * xs + b * ys + c
        yin = d * xs + e * ys + f
        ok = (xin >= 0) & (xin < W) & (yin >= 0) & (yin < H)
        xi = xin.floor().clamp(0, W - 1).long()
        yi = yin.floor().clamp(0, H - 1).long()
        out = img[yi, xi]
        out[~ok] = 0
        return out.contiguous()

    @_on_own_device
    def views_on_device(self, img: torch.Tensor, rects, clahe: bool, filter: str = "bilinear"):
        """img: u8 [H,W,3] on the device.  rects: (x0,y0,x1,y1) crops, or "bicubic" = the whole image resized to S x S with
        PIL's bicubic filter.  Returns (model input u8 [V,S,S,3], gray256 f32 [V,256,256])."""
        S = self.arch.image_size
        xs, gs = [], []
        for r in rects:
            if r == "bicubic":
                v = ops.resize_u8(img[None], S, S, "bicubic")            # pil.resize((S,S), BICUBIC); Resize((S,S)) is then the identity
                xs.append(v)
                gs.append(ops.gray256_from_rgb(v, clahe))
            else:
                x0, y0, x1, y1 = r
                crop = img[y0:y1, x0:x1][None]        # a view: the kernels take the rectangle's base pointer and strides
                xs.append(crop.contiguous() if crop.shape[1:3] == (S, S) else ops.resize_u8(crop, S, S, filter))
                gs.append(ops.gray256_from_rgb(crop, clahe))
        return torch.cat(xs, 0), torch.cat(gs, 0)

    def _upload(self, pil_or_array) -> torch.Tensor:
        """One pinned H2D copy of the original pixels (u8 [H,W,3])."""
        if isinstance(pil_or_array, torch.Tensor):
            t = pil_or_array
        else:
            arr = np.asarray(pil_or_array.convert("RGB") if hasattr(pil_or_array, "convert") else pil_or_array, dtype=np.uint8)
            t = torch.from_numpy(np.ascontiguousarray(arr))
        if not t.is_cuda:
            t = t.pin_memory().to(self.device, non_blocking=True)
        return t.contiguous()

    @torch.no_grad()
    @_on_own_device
    def detect_core_device(self, images, views: Optional[str] = "v2", rot90: bool = False, clahe: bool = False,
                           freq_temp: float = 1.25):
        """`detect_core` for a list of images with every view produced on the device.
        views "v2" = the 6 views of deepfake-detector-v2/app.py:1418-1430, "v3" = the 9 crops of appv3.py:3315-3350,
        None = single view (multicrop=False).  rot90 adds appv3's dual-view stabiliser (:3239-3249):
        p_sig = 0.6 sigma(z_sig) + 0.4 sigma(z_rot90), z_sig = logit(p_sig).  One engine batch for everything."""
        S = self.arch.image_size
        xs, gs, wts, counts = [], [], [], []
        for im in images:
            img = self._upload(im)
            H, W = img.shape[:2]
            if views == "v2":
                rects, w = self.multicrop_rects_v2(W, H)
            elif views == "v3":
                rects, w = self.multicrop_rects_v3(W, H)
            else:
                rects, w = [(0, 0, W, H)], [1.0]
            x, g = self.views_on_device(img, rects, clahe)
            if rot90:   # model input only: the frequency branch does not look at the rotated view
                xr = ops.resize_u8(self.rotate90_noexpand(img)[None], S, S, "bilinear") if (H, W) != (S, S) \
                    else self.rotate90_noexpand(img)[None]
                x = torch.cat([x, xr], 0)
            xs.append(x)
            gs.append(g)
            wts.append(w)
            counts.append(len(w))
        x_all, g_all = torch.cat(xs, 0), torch.cat(gs, 0)
        pooled, _ = self.engine(x_all)
        z_all = ops.head_fwd(self.head, pooled)[1]
        zf_all = self.scoring(torch.zeros(g_all.shape[0], device=self.device), feats=self.freq.from_gray(g_all))["z_freq"]
        zs, zf, o, of = [], [], 0, 0
        for w in wts:   # a handful of scalars per image: combined with torch ops on the device, no host round trip
            wt = torch.tensor(w, dtype=torch.float32, device=self.device)
            n = len(w)
            z = (z_all[o:o + n] * wt).sum()
            if rot90:
                p = 0.6 * torch.sigmoid(z) + 0.4 * torch.sigmoid(z_all[o + n])
                p = p.clamp(1e-6, 1 - 1e-6)
                z = torch.log(p / (1 - p))
            zs.append(z)
            zf.append((zf_all[of:of + n] * wt).sum())
            o += n + (1 if rot90 else 0)
            of += n
        out = self.scoring(torch.stack(zs).contiguous(), z_freq=torch.stack(zf).contiguous())
        host = {k: v.cpu().numpy() for k, v in out.items()}
        res = []
        for i in range(len(images)):
            zsi, zfi = float(host["z_sig"][i]), float(host["z_freq"][i])
            res.append({"z_sig": zsi, "z_freq": zfi, "z_scaled": float(host["z_scaled"][i]),
                        "p_fake_raw": float(host["p_raw"][i]), "p_fake_coral": float(host["p_coral"][i]),
                        "p_blend": float(host["p_blend"][i]), "visual_prob": 1.0 / (1.0 + np.exp(-zsi)),
                        "freq_prob": 1.0 / (1.0 + np.exp(-zfi / freq_temp)), "p_or": None, "p_moe": None,
                        "risk_idx": int(host["risk_idx"][i]), "risk_probs": torch.from_numpy(host["risk_probs"][i].copy()),
                        "entropy": float(host["entropy"][i])})
        return res

    @torch.no_grad()
    @_on_own_device
    def patch_grid(self, image, rows: int = 4, cols: int = 4, clahe: bool = False, min_side: int = 64):
        """`compute_patch_grid` (deepfake-detector-v2/app.py:1461-1485): p_fake_raw of every grid cell, all rows x cols cells
        of the image in ONE batch (the reference runs one batch-1 detect_core per cell).  Returns (grid [rows,cols] f32,
        flat list) or (None, []) for images below MIN_SIDE."""
        img = self._upload(image)
        H, W = img.shape[:2]
        rects = self.patch_grid_rects(W, H, rows, cols, min_side)
        if rects is None:
            return None, []
        live = [r for r in rects if r is not None]
        grid = np.zeros((rows, cols), np.float32)
        if live:
            x, g = self.views_on_device(img, live, clahe)
            pooled, _ = self.engine(x)
            z_sig = ops.head_fwd(self.head, pooled)[1]
            p = self.scoring(z_sig, feats=self.freq.from_gray(g))["p_raw"].cpu().numpy()
            it = iter(p)
            for i, r in enumerate(rects):
                if r is not None:
                    grid[i // cols, i % cols] = next(it)
        return grid, [float(v) for v in grid.reshape(-1)]

    @torch.no_grad()
    @_on_own_device
    def frame_features(self, frames: torch.Tensor, filter: str = "bilinear") -> torch.Tensor:
        """Video path (hidf_video_classifier.py:299-320): u8 frames [F,H,W,3] (host or device, one upload) -> L2-normalised
        per-frame embeddings f32 [F,D]; `frame_features(...).mean(0)` is the reference's temporal average pool."""
        S = self.arch.image_size
        fr = self._upload(frames)
        if tuple(fr.shape[1:3]) != (S, S):
            fr = ops.resize_u8(fr, S, S, filter)
        pooled, _ = self.engine(fr)
        return ops.head_fwd(ops.HeadParams(0, self.arch.hidden_size, 0.0, self.device), pooled, want_features=True)[0]

    # ---- host-buffer path (what a caller of the reference loops sees) -----------------------------------
    @_on_own_device
    def detect(self, images_host: torch.Tensor, gray256_host: Optional[torch.Tensor] = None, resize_mode: int = 0,
               clahe: bool = True, pil_resize: Optional[str] = None) -> np.ndarray:
        """Host (ideally pinned) u8 NHWC images [+ f32 gray256; None = computed on the device from the same
        pixels] -> numpy [B,14] score records.  An empty batch gives an empty [0,14] array (the reference's loops simply do not
        iterate); the C ABI itself rejects B = 0 with DFD_ERR_SHAPE."""
        if images_host.shape[0] == 0:
            return np.zeros((0, len(PACKED_FIELDS)), dtype=np.float32)
        img = images_host.to(self.device, non_blocking=True)
        gray = None if gray256_host is None else gray256_host.to(self.device, non_blocking=True)
        packed = self.pack(self.detect_device(img, gray, resize_mode, clahe, pil_resize))
        key = f"out{packed.shape[0]}"
        if key not in self._pin:
            self._pin[key] = torch.empty(packed.shape, dtype=torch.float32).pin_memory()
        self._pin[key].copy_(packed, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        # a fresh array per call: the pinned buffer is reused by the next call of the same batch size, and callers collect
        # per-batch results (`all_probs.extend(...)` in the reference loops) — 28 KB per 512 images
        return self._pin[key].numpy().copy()

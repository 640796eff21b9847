"""Attention-map timing on one B200 (CUDA events): the forward with the attention tap off, in head-mean and in per-head
mode; the attention_probs kernel on its own with bytes and FLOPs from shapes and its share of the binding roofline; the
rollout's HBM rate; DetectionPipeline.explain() images/s.  Writes one JSON document (--out) with the card and its power
limit read in the same run.  Peaks as scripts/kbench.py takes them: MEASURED_PEAKS.json if present, else 1384.8 TF/s
sustained bf16 and 6545.9 GB/s HBM."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dfd import ops  # noqa: E402
from dfd.engine import ARCHS, SiglipEngine  # noqa: E402
from oracle import siglip_ref as R  # noqa: E402

DEV = "cuda:0"
PEAKS = {"bf16_tflops_sustained": 1384.8, "hbm_gbs": 6545.9}
try:
    PEAKS.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
except Exception:
    pass


def timeit(fn, iters, warm=2):
    """Median ms of `iters` CUDA-event-timed calls after `warm` untimed ones."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def probs_roofline(B, N, H, hd, per_head, ms):
    """bytes and FLOPs the kernel needs, from shapes: qkv q|k read once, P written once; two Q·Kᵀ sweeps."""
    read = B * N * 2 * H * hd * 2
    write = 4 * B * N * N * (H if per_head else 1)
    flops = 2 * (2.0 * B * H * N * N * hd)
    t_bytes = (read + write) / (PEAKS["hbm_gbs"] * 1e9)
    t_flops = flops / (PEAKS["bf16_tflops_sustained"] * 1e12)
    bound = "hbm" if t_bytes >= t_flops else "tensor"
    return {"ms": ms, "bytes": read + write, "flops": flops, "gb_s": (read + write) / ms / 1e6,
            "tflop_s": flops / ms / 1e9, "exp_per_s": 2.0 * B * H * N * N / ms * 1e3, "roofline_bound": bound,
            "share_of_roofline": max(t_bytes, t_flops) * 1e3 / ms}


def run(name, B, B_per_head, iters):
    c = R.CONFIGS[name]
    a = ARCHS[name]
    L, H, N, hd = a.num_hidden_layers, a.num_attention_heads, a.tokens, a.head_dim
    eng = SiglipEngine(a, 0, max_batch=B, fuse_ln=True).load_state_dict(R.init_state_dict(c, 0))
    img = R.synthetic_images(B, c.image_size, 0).to(DEV)
    res = {"B": B, "tokens": N, "layers": L, "heads": H}
    fwd = timeit(lambda: eng.forward(img), iters)
    eng.profile(iters + 2)
    timeit(lambda: eng.forward(img), iters, warm=0)
    fam = eng.profile_read()
    eng.profile(0)
    res["forward_ms"] = fwd
    res["forward_attention_ms"] = fam["attention"][0] / iters
    res["forward_tap_mean_ms"] = timeit(lambda: eng.forward_attentions(img), iters)
    imgp = img[:B_per_head]
    res["per_head_B"] = B_per_head
    res["forward_ms_at_per_head_B"] = timeit(lambda: eng.forward(imgp), iters)
    res["forward_tap_per_head_ms"] = timeit(lambda: eng.forward_attentions(imgp, per_head=True), iters)

    g = torch.Generator(device=DEV).manual_seed(0)
    qkv = torch.randn(B * N, 3 * H * hd, device=DEV, generator=g).to(torch.bfloat16)
    res["probs_mean"] = probs_roofline(B, N, H, hd, False, timeit(
        lambda: ops.attention_probs(qkv, B, N, H, hd, per_head=False), iters))
    qkvp = qkv[:B_per_head * N]
    res["probs_per_head"] = probs_roofline(B_per_head, N, H, hd, True, timeit(
        lambda: ops.attention_probs(qkvp, B_per_head, N, H, hd, per_head=True), iters))
    res["attention_flash_ms"] = timeit(lambda: ops.attention_bf16(qkv, B, N, H, hd), iters)

    _, attn, map_p = eng.forward_attentions(img)
    roll = timeit(lambda: ops.attention_rollout(attn, map_p, 0.5, a.image_size), iters)
    rb = 4.0 * L * B * N * N
    res["rollout"] = {"ms": roll, "bytes": rb, "gb_s": rb / roll / 1e6, "share_of_hbm": rb / roll / 1e6 / PEAKS["hbm_gbs"]}
    del attn
    eng.close()

    from dfd.pipeline import DetectionPipeline
    from dfd.scoring import ScoringStack
    from oracle import scoring_ref as S

    st = ScoringStack(DEV, S.init_freq_mlp_g2(2), S.init_fusion_g2(3), [-1.0, -0.2, 0.3, 1.5], 1.0)
    pipe = DetectionPipeline(name, R.init_state_dict(c, 0), R.init_head("B", c.hidden_size, 1), st, 0, max_batch=B)
    ex = timeit(lambda: pipe.explain(img), iters)
    res["explain_ms"] = ex
    res["explain_images_per_s"] = B / ex * 1e3
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="tiny shapes: checks the script end to end, times nothing useful")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_maps_bench.py needs a GPU")
    doc = {"card": card(), "peaks": PEAKS}
    if args.quick:
        doc["small-hd72"] = run("small-hd72", 4, 2, 2)
    else:
        doc["so400m-384"] = run("siglip2-so400m-patch14-384", 64, 8, args.iters)
        doc["base-224"] = run("siglip2-base-patch16-224", 256, 64, args.iters)
    txt = json.dumps(doc, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(txt + "\n")


if __name__ == "__main__":
    main()

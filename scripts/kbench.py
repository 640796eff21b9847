"""Kernel-level timing on one B200 (CUDA events, L2 flushed between iterations). Not the driver's bench —
a development aid: prints TFLOP/s or GB/s per kernel and per shape, against MEASURED_PEAKS.json."""
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dfd import engine, ops  # noqa: E402

DEV = "cuda:0"
PEAKS = {"bf16_tflops": 1639.8, "bf16_tflops_sustained": 1384.8, "hbm_gbs": 6545.9}
try:
    PEAKS.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
except Exception:
    pass
_flush = None


def flush_l2():
    global _flush
    if _flush is None:
        _flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    _flush.zero_()


def timeit(fn, iters=5, warm=2, flush=True):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush:
            flush_l2()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def gemms(B, arch):
    N, D, I = arch.tokens, arch.hidden_size, arch.intermediate_size
    M = B * N
    shapes = [("qkv", M, 3 * D, D, {}), ("out+res", M, D, D, {"res": True}), ("fc1+gelu", M, I, D, {"act": 1}),
              ("fc2+res", M, D, I, {"res": True}), ("patch", M, D, (3 * arch.patch_size ** 2 + 63) // 64 * 64, {})]
    for name, m, n, k, o in shapes:
        a = torch.randn(m, k, device=DEV).to(torch.bfloat16)
        w = (torch.randn(n, k, device=DEV) / math.sqrt(k)).to(torch.bfloat16)
        bias = torch.randn(n, device=DEV)
        out = torch.empty(m, n, dtype=torch.bfloat16, device=DEV)
        res = torch.randn(m, n, device=DEV).to(torch.bfloat16) if o.get("res") else None
        for tn in (1256, 2128, 2192, 2256, 0):
            med, best = timeit(lambda: ops.gemm_bf16(a, w, bias=bias, act=o.get("act", 0), residual=res, out=out, tile_n=tn))
            tf = 2.0 * m * n * k / med / 1e9
            print(f"gemm {name:9s} M={m} N={n} K={k} tile={tn:4d}: {med:8.3f} ms  {tf:7.1f} TF/s "
                  f"({tf / PEAKS['bf16_tflops'] * 100:4.1f}% of measured burst)  best {best:.3f}", flush=True)
        med, _ = timeit(lambda: torch.matmul(a, w.t(), out=out))
        print(f"   cuBLAS (torch.matmul, no epilogue) {med:8.3f} ms {2.0 * m * n * k / med / 1e9:7.1f} TF/s", flush=True)
        del a, w, out, res


def attention(B, arch):
    N, H, hd = arch.tokens, arch.num_attention_heads, arch.head_dim
    qkv = torch.randn(B * N, 3 * H * hd, device=DEV).to(torch.bfloat16)
    fl = 4.0 * N * N * H * hd * B
    for impl in (2, 5):
        med, best = timeit(lambda: ops.attention_bf16(qkv, B, N, H, hd, impl=impl))
        print(f"attention impl={impl} B={B} N={N} H={H} hd={hd}: {med:8.3f} ms {fl / med / 1e9:7.1f} TF/s best {best:.3f}", flush=True)
    try:
        q, k, v = (qkv[:, i * H * hd:(i + 1) * H * hd].reshape(B, N, H, hd).transpose(1, 2) for i in range(3))
        med, _ = timeit(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v))
        print(f"   torch SDPA {med:8.3f} ms {fl / med / 1e9:7.1f} TF/s", flush=True)
    except Exception as e:  # noqa: BLE001
        print("   torch SDPA failed:", e)
    x = torch.randn(B * N, H * hd, device=DEV).to(torch.bfloat16)
    g = torch.ones(H * hd, device=DEV)
    med, _ = timeit(lambda: ops.layernorm_bf16(x, g, g))
    by = x.numel() * 4
    print(f"layernorm M={B * N} D={H * hd}: {med:8.3f} ms {by / med / 1e6:7.1f} GB/s "
          f"({by / med / 1e6 / PEAKS['hbm_gbs'] * 100:4.1f}% of measured)", flush=True)


def memory_bound(B, arch):
    """HBM-bound kernels of the detect step: algorithmic bytes (DESIGN.md §3) / CUDA-event time, L2 flushed."""
    from dfd import scoring

    S, P, D, N, H = arch.image_size, arch.patch_size, arch.hidden_size, arch.tokens, arch.num_attention_heads
    peak = PEAKS["hbm_gbs"]

    def line(name, by, fn):
        med, best = timeit(fn, iters=7)
        print(f"{name:34s} {med:7.3f} ms  {by / 1e6:9.1f} MB  {by / med / 1e6:7.1f} GB/s ({by / med / 1e6 / peak * 100:4.1f}% of measured HBM)",
              flush=True)

    img = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, device=DEV)
    lda = (3 * P * P + 63) // 64 * 64
    line(f"patchify B={B} S={S}", B * (3 * S * S + N * lda * 2), lambda: ops.patchify(img, S, P))
    x = torch.randn(B * N, D, device=DEV).to(torch.bfloat16)
    g = torch.ones(D, device=DEV)
    line(f"layernorm M={B * N} D={D}", x.numel() * 4, lambda: ops.layernorm_bf16(x, g, g))
    kv = torch.randn(B * N, 2 * D, device=DEV).to(torch.bfloat16)
    q = torch.randn(D, device=DEV)
    line(f"map_attention B={B} N={N}", kv.numel() * 2, lambda: ops.map_attention_bf16(kv, q, B, N, H, D // H))
    scratch = torch.empty(ops._lib.load().dfd_gray256_scratch_bytes(B, S, S), dtype=torch.uint8, device=DEV)
    out = torch.empty(B, 256, 256, device=DEV)
    for clahe in (False, True):
        # RGB in, gray256 out, plus the u8 intermediates written and read once each (luma [, CLAHE], row pass)
        inter = S * S * (2 if clahe else 1) + 256 * S
        line(f"gray256 B={B} S={S} clahe={clahe}", B * (3 * S * S + 2 * inter + 256 * 256 * 4),
             lambda: ops.gray256_from_rgb(img, clahe, scratch, out))
    luts = scoring.build_freq_luts(torch.device(DEV))
    fscr = torch.empty(ops._lib.load().dfd_freq_scratch_bytes(B), dtype=torch.uint8, device=DEV)
    line(f"freq_features B={B}", B * (256 * 256 * 4 + 2 * 256 * 129 * 8 + 96), lambda: ops.freq_features(out, luts, scratch=fscr))


def full(name, B, iters=3, fuse_ln=False):
    from dfd import weights

    arch = engine.ARCHS[name]
    eng = engine.SiglipEngine(arch, 0, max_batch=B, fuse_ln=fuse_ln).load_state_dict(weights.random_vision_state_dict(arch, 0, DEV))
    img = torch.randint(0, 256, (B, arch.image_size, arch.image_size, 3), dtype=torch.uint8, device=DEV)
    med, best = timeit(lambda: eng(img), iters=iters, warm=2, flush=False)
    tf = arch.flops_per_image() * B / med / 1e9
    print(f"engine {name} B={B} fuse_ln={fuse_ln}: {med:9.3f} ms  {B / med * 1e3:9.1f} img/s  {tf:7.1f} TF/s "
          f"({tf / PEAKS['bf16_tflops_sustained'] * 100:4.1f}% of measured sustained) ws={eng.workspace_bytes / 2**30:.2f} GiB",
          flush=True)
    eng.close()


if __name__ == "__main__":
    what = sys.argv[1:] or ["gemm", "attn", "full"]
    so, ba = engine.ARCHS["siglip2-so400m-patch14-384"], engine.ARCHS["siglip2-base-patch16-224"]
    if "gemm" in what:
        gemms(64, so)
        gemms(256, ba)
    if "attn" in what:
        attention(64, so)
        attention(256, ba)
    if "mem" in what:
        memory_bound(512, so)
        memory_bound(256, ba)
    if "full" in what:
        for f in (False, True):
            full("siglip2-base-patch16-224", 256, fuse_ln=f)
            full("siglip2-so400m-patch14-384", 128, fuse_ln=f)

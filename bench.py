#!/usr/bin/env python
"""bench.py — images/sec of the detection hot path (SigLIP-2 so400m/14-384 backbone + classifier head + FreqMLP
features + fusion/CORAL epilogue) on N B200s, data parallel.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (N>1: launched by torchrun)
    python bench.py --impl reference [--gpus N] --steps K --warmup W  # the reference's CPU path on the host cores

One "step" = one pass of the whole hot path over one batch of synthetic images per GPU (BASELINE.json
configs[2]: so400m-patch14-384, 729 tokens, batch 512 per GPU, weak scaling).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec SigLIP-2 so400m/14-384 detect"           # BASELINE.json:metric (the default workload)
METRICS = {"so400m-384": METRIC, "base-224": "images/sec SigLIP-2 base-patch16-224 detect"}
WORKLOADS = {
    "so400m-384": ("google/siglip2-so400m-patch14-384", 512),
    "base-224": ("google/siglip2-base-patch16-224", 256),
}


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks.update(json.load(f))
        peaks["source"] = "measured"
    except Exception:
        pass
    return peaks


def load_traffic():
    """dram bytes per GEMM launch (dram__bytes_read.sum + dram__bytes_write.sum averaged over the 113 GEMM launches of one step)
    from the committed ncu capture of this command, profiles/r02_gemm_traffic.json; None if absent.  Reported beside
    `roofline.traffic` (which stays null unless --gemm-traffic is given): it was not measured in this run."""
    for name in ("r02_gemm_traffic.json", "gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return {"dram_bytes_per_launch": float(json.load(f)["dram_bytes_per_launch"]), "source": "profiles/" + name}
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.t = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            if len(p) >= 7:
                self.rows.append(p)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for p in self.rows:
            try:
                sm.append(float(p[0]))
                mx = float(p[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# CPU arms (the only places bench.py touches oracle/): cpu_baseline of our arm, and --impl reference
# ---------------------------------------------------------------------------------------------------------
class CpuReference:
    """The reference's CPU path for the hot path: backbone = the library call the reference makes
    (transformers.SiglipVisionModel, Siglip2sidafrozen.py:753,787; fp32, all host threads) when importable, else
    the oracle restatement; heads / frequency features / fusion / CORAL = the oracle port of the reference's
    functions (train_fusion_head_only.py:142-317, app.py:1265-1396), one image at a time like its loops."""

    def __init__(self, workload: str):
        import torch

        from oracle import scoring_ref as S
        from oracle import siglip_ref as R

        self.torch, self.S, self.R = torch, S, R
        name = WORKLOADS[workload][0].split("/")[-1]
        self.cfg = R.CONFIGS[name]
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        sd = R.init_state_dict(self.cfg, 0)
        self.sd, self.hf, self.kind = sd, None, "port"
        try:
            from transformers import SiglipVisionConfig, SiglipVisionModel

            c = self.cfg
            m = SiglipVisionModel(SiglipVisionConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                                                     num_hidden_layers=c.num_hidden_layers,
                                                     num_attention_heads=c.num_attention_heads,
                                                     image_size=c.image_size, patch_size=c.patch_size)).eval()
            m.load_state_dict({"vision_model." + k: v for k, v in sd.items()}, strict=True)
            self.hf = m
        except Exception:
            self.hf = None
        self.head = R.init_head("B", self.cfg.hidden_size, 1)
        self.fm, self.fu = S.init_freq_mlp_g2(2), S.init_fusion_g2(3)
        self.cuts = __import__("numpy").array([-1.0, -0.2, 0.3, 1.5], dtype="float32")

    def run(self, n: int, seed: int = 0) -> float:
        """Hot path over n synthetic images; returns seconds."""
        import numpy as np

        torch, S, R = self.torch, self.S, self.R
        img = R.synthetic_images(n, self.cfg.image_size, seed)
        t0 = time.perf_counter()
        with torch.inference_mode():
            x = R.preprocess_u8(img)
            if self.hf is not None:
                pooled = self.hf(pixel_values=x).pooler_output
            else:
                pooled = R.siglip_vision_forward(self.sd, self.cfg, x, "fp32")["pooler_output"]
            z_sig = R.classifier_head(self.head, "B", pooled, 1e-6).numpy()
        feats = np.stack([S.extract_freq_vector(S.gray256_from_rgb_u8(im.numpy(), True)) for im in img])
        z = S.fusion_g2(self.fu, S.freq_mlp_g2(self.fm, feats), z_sig)
        S.detect_scores(z, self.cuts, 1.0)
        return time.perf_counter() - t0

    def describe(self, n: int) -> str:
        bb = "transformers.SiglipVisionModel fp32 (the reference's own backbone call)" if self.hf is not None \
            else "oracle/siglip_ref.py fp32"
        return (f"{n} synthetic {self.cfg.image_size}x{self.cfg.image_size} images per step: backbone {bb}, "
                f"{self.cores} torch threads; heads+freq features+fusion+CORAL = oracle port, single thread per image")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference(args.workload)
    t1 = ref.run(1, seed=99)                       # probe (also first-touch warm-up)
    n = max(1, min(16, int(4.0 / max(t1, 1e-3))))  # ~4 s per step
    for _ in range(args.warmup):
        ref.run(n, seed=1)
    ts = [ref.run(n, seed=2 + i) for i in range(args.steps)]
    total = sum(ts)
    value = n * args.steps / total
    line = {"impl": "reference", "metric": METRICS.get(args.workload, METRIC), "value": value, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload][0]} detect, CPU sample of {n} images/step"},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": ref.cores, "kind": ref.kind,
                             "sample": ref.describe(n)},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def hbm_entry(name, bytes_per_image, images, ms, calls, peak):
    if not calls or ms <= 0:
        return None
    ach = bytes_per_image * images / (ms / 1e3) / 1e9
    return {"kernel": name, "bound": "hbm", "algorithmic_bytes_per_image": int(bytes_per_image), "images": int(images),
            "calls": calls, "avg_ms": ms / calls, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}


def unit_plan(total_images: int, world: int, B: int, sub: int):
    """The work queue's units as (first image, images).  One GPU: whole batches.  Several GPUs: `sub`-image units for the bulk
    of the work, then a tail of half- and quarter-size units (2 x world of each), so that the ranks finish within a quarter
    unit of each other instead of a whole one (guided self-scheduling; sizes stay aligned to their offsets)."""
    if world == 1 or sub >= B and world == 1:
        return [(o, min(sub, total_images - o)) for o in range(0, total_images, sub)]
    sizes = [sub // 2, sub // 4] if sub >= 4 and sub % 4 == 0 else []
    tail = sum(sz * 2 * world for sz in sizes)
    plan, off = [], 0
    while total_images - off >= tail + sub:
        plan.append((off, sub))
        off += sub
    for sz in sizes:
        for _ in range(2 * world):
            if total_images - off >= sz:
                plan.append((off, sz))
                off += sz
    while off < total_images:
        sz = min(sizes[-1] if sizes else sub, total_images - off)
        plan.append((off, sz))
        off += sz
    return plan


def dump_records(out_dir: str, records) -> None:
    """Score records [n, 14] of one step -> out_dir/<field>.npy (float32), the fields DetectionPipeline.detect_device
    returns (risk_probs as [n, 5]).  The bench's weights and images are seeded, so two builds can be compared field by field."""
    import numpy as np

    from dfd import pipeline

    os.makedirs(out_dir, exist_ok=True)
    rec = records.float().cpu().numpy()
    fields = pipeline.PACKED_FIELDS
    n_scalar = fields.index("risk_p0")
    for i, name in enumerate(fields[:n_scalar]):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(rec[:, i]))
    np.save(os.path.join(out_dir, "risk_probs.npy"), np.ascontiguousarray(rec[:, n_scalar:]))


def seeded_workload(arch, B: int, local: int, max_batch: int, fuse_ln: bool = True, precise_residual: bool = False,
                    graphs: bool = True):
    """The pipeline the bench times (seeded random weights of `arch`) and its B seeded u8 images on cuda:local.  Every rank
    draws the same images: the records of a work-queue unit do not depend on which rank took it."""
    import torch

    from dfd import pipeline, scoring, weights

    dev = torch.device("cuda", local)
    bsd = weights.random_vision_state_dict(arch, seed=0, device=dev)
    st = scoring.ScoringStack(dev, weights.random_freq_mlp_g2(2), weights.random_fusion_g2(3), [-1.0, -0.2, 0.3, 1.5], 1.0)
    pipe = pipeline.DetectionPipeline(arch, bsd, weights.random_classifier_head("B", arch.hidden_size, 1), st, device=local,
                                      max_batch=max_batch, fuse_ln=fuse_ln, precise_residual=precise_residual, graphs=graphs)
    del bsd
    S = arch.image_size
    g = torch.Generator(device=dev).manual_seed(1234)
    images = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, device=dev, generator=g)
    return pipe, images


def run_ours(args):
    import torch

    from dfd import _lib, distributed, pipeline
    from dfd.engine import ARCHS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the dfd hot path has no CPU fallback")
    rank, world, local = distributed.init_from_env("nccl")
    if world != args.gpus and world > 1:
        print(f"bench.py: WORLD_SIZE={world} overrides --gpus {args.gpus}", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    arch_name, default_batch = WORKLOADS[args.workload]
    B = args.batch or default_batch
    strong = args.global_batch > 0
    if strong:   # strong scaling (SURVEY.md §8d): the global batch is fixed, every GPU holds its share of it
        B = max(1, args.global_batch // world)
    arch = ARCHS[arch_name]
    peaks = load_peaks()
    lib = _lib.load()
    # sub-batch = the unit of the work queue.  One GPU: the whole batch in one call.  Several GPUs: halves of the per-GPU batch
    # (256 images run within 0.1 % of a 512-image call, 128 cost 0.6 %), with a tail of shorter units (unit_plan).
    sub = args.sub_batch or (B if (world == 1 or strong) else max(1, B // 2))
    sub = min(sub, B)

    pipe, images = seeded_workload(arch, B, local, max_batch=min(sub, args.max_batch), fuse_ln=bool(args.fuse_ln),
                                   precise_residual=bool(args.precise_residual), graphs=bool(args.graphs))
    S = arch.image_size
    F = len(pipeline.PACKED_FIELDS)

    def unit_images(unit, src):
        off, n = unit
        lo = off % B                       # every rank holds B resident images; a unit is a slice of them
        return src[lo: lo + n] if lo + n <= B else src[:n]

    def drain_device(plan, key: str, slab):
        """This rank's share of the queue of units `plan`, inputs resident in HBM; the records of unit (off, n) land in
        slab[off : off + n].  Returns (units, images) taken."""
        q = distributed.WorkQueue(key)
        inflight, done, imgs = [], 0, 0
        while True:
            # claim only when at most one unit is still outstanding on the device (the host stays at most two units ahead): a rank
            # that claimed first and waited afterwards held up to three units — at the end of the queue those are tail units a
            # faster GPU could have taken (8 GPUs, 5 steps: 65-71 ms of 1.67 s waiting at the final collective)
            while len(inflight) >= 2:
                inflight.pop(0).synchronize()
            u = q.next()
            if u >= len(plan):
                break
            off, n = plan[u]
            slab[off: off + n] = pipe.pack(pipe.detect_device(unit_images(plan[u], images), None, clahe=True))
            ev = torch.cuda.Event()
            ev.record()
            inflight.append(ev)
            done += 1
            imgs += n
        return done, imgs

    def gather(slab):
        # every unit was filled by exactly one rank and is zero elsewhere: a sum over ranks IS the all-gather of the score
        # records under dynamic ownership (x + 0 is exact) — ONE collective for all steps, not a rendezvous per step
        if world > 1:
            distributed.all_reduce_sum_(slab)
        return slab

    warm = max(args.warmup, 3)
    per_step = world * B
    slab = torch.zeros((warm * per_step, F), dtype=torch.float32, device=dev)
    t_w = time.perf_counter()
    drain_device(unit_plan(warm * per_step, world, B, sub), "dfd_bench_warm", slab)
    gather(slab)
    torch.cuda.synchronize()
    # short steps (base-224: 10 ms) would start the timed region while the clocks are still ramping: warm up for at least ~1.5 s
    step_s = max((time.perf_counter() - t_w) / warm, 1e-4)
    extra = int(distributed.max_over_ranks(max(0.0, 1.5 - warm * step_s) / step_s, dev))
    if extra > 0:
        slab = torch.zeros((extra * per_step, F), dtype=torch.float32, device=dev)
        drain_device(unit_plan(extra * per_step, world, B, sub), "dfd_bench_warm2", slab)
        gather(slab)
        torch.cuda.synchronize()
        warm += extra

    # ---- timed region 1: inputs resident in HBM ------------------------------------------------------
    # no instrumentation inside: the engine forward runs as it does in production (CUDA-graph replay when --graphs 1)
    plan = unit_plan(args.steps * per_step, world, B, sub)
    slab = torch.zeros((args.steps * per_step, F), dtype=torch.float32, device=dev)
    sampler = ClockSampler(local)
    launches0 = lib.dfd_launch_count()
    replays0 = pipe.engine.graph_replays
    distributed.barrier()
    torch.cuda.synchronize()
    e0, eb, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    mine, mine_images = drain_device(plan, "dfd_bench_timed", slab)
    eb.record()                      # this rank's own kernels end here; what follows is waiting for the others
    gather(slab)
    e1.record()
    distributed.barrier()
    torch.cuda.synchronize()
    dt = distributed.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
    launches = lib.dfd_launch_count() - launches0
    replays = pipe.engine.graph_replays - replays0
    clocks = sampler.stop()
    value = world * B * args.steps / dt
    if args.dump_outputs and rank == 0:      # after gather(): the slab holds every rank's records
        dump_records(args.dump_outputs, slab[(args.steps - 1) * per_step:])

    # ---- profiled pass (not part of `value`): the same work with every launch of the engine bracketed by CUDA events on its
    # stream (eager launches), read back once at the end — per-family / per-GEMM-type durations for the roofline entries
    slab_p = torch.zeros((args.steps * per_step, F), dtype=torch.float32, device=dev)
    chunks_per_unit = (sub + pipe.engine.max_batch - 1) // pipe.engine.max_batch
    pipe.engine.profile(len(plan) * chunks_per_unit)   # room for the case that this rank takes every unit
    pipe.profile_stages(True)
    distributed.barrier()
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    _, images_p = drain_device(plan, "dfd_bench_profiled", slab_p)
    p1.record()
    torch.cuda.synchronize()
    fam_all = pipe.engine.profile_read(by_gemm_type=True)
    fam = {k: v for k, v in fam_all.items() if not k.startswith("gemm_")}
    stages = pipe.profile_stages_read()
    pipe.profile_stages(False)
    pipe.engine.profile(0)
    prof_busy_ms = p0.elapsed_time(p1)
    distributed.barrier()
    del slab_p
    mine_rec = {"rank": rank, "units": mine, "images": mine_images, "busy_ms": e0.elapsed_time(eb),
                "wait_ms": eb.elapsed_time(e1), "graph_replays": replays,
                "profiled_pass": {"images": images_p, "busy_ms": prof_busy_ms,
                                  "kernel_ms": sum(v[0] for v in fam.values()) + sum(v[0] for v in stages.values())},
                "sm_mhz": clocks.get("sm_mhz"), "reasons": clocks.get("reasons")}
    per_rank = [mine_rec]
    if world > 1:
        import torch.distributed as dist

        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine_rec)

    # ---- timed region 2: end to end through the public API, host buffers --------------------------------
    # DetectionPipeline.detect_many: pinned host images in, numpy score records out; the upload of sub-batch k+1 and the
    # download of k's records run on a copy stream under k's kernels.  Same work queue.
    h_img = torch.empty((B, S, S, 3), dtype=torch.uint8).pin_memory()
    h_img.copy_(images)

    def drain_host(plan_h, key: str):
        q = distributed.WorkQueue(key)
        taken = []

        def feed():
            while True:
                u = q.next()
                if u >= len(plan_h):
                    return
                taken.append(plan_h[u])
                yield unit_images(plan_h[u], h_img)

        recs = pipe.detect_many(feed(), clahe=True)
        total = plan_h[-1][0] + plan_h[-1][1]
        out = torch.zeros((total, F), dtype=torch.float32)
        for (off, n), r in zip(taken, recs):
            out[off: off + n] = torch.from_numpy(r)
        if world > 1:   # the all-gather of the records (dynamic ownership, see gather())
            out = gather(out.to(dev)).cpu()
        return out, sum(r.shape[0] for r in recs)

    drain_host(unit_plan(4 * per_step, world, B, sub), "dfd_bench_e2e_warm")   # every input slab of detect_many seen twice: graphs captured
    distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec, n_mine = drain_host(plan, "dfd_bench_e2e")
    torch.cuda.synchronize()
    dt_e2e = distributed.max_over_ranks(time.perf_counter() - t0, dev)
    distributed.barrier()
    e2e_value = world * B * args.steps / dt_e2e
    # bytes this rank moved per step (rank 0's share; the ranks' shares differ by the dynamic split)
    h2d = n_mine * S * S * 3 // args.steps
    d2h = n_mine * F * 4 // args.steps

    if rank != 0:
        return
    step_ms = dt / args.steps * 1e3
    busy_ms = prof_busy_ms                   # shares and achieved rates below refer to rank 0's profiled pass
    my_images = max(images_p, 1)
    roof, hbm = None, []
    if fam["gemm"][0] > 0:
        gemm_flops = pipe.engine.gemm_flops(1) * my_images
        ach = gemm_flops / (fam["gemm"][0] / 1e3) / 1e12
        peak = float(peaks["bf16_tflops_sustained"])
        shares = {k: v[0] / busy_ms for k, v in fam.items()}
        shares.update({k: v[0] / busy_ms for k, v in stages.items()})
        roof = {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel (all GEMM launches of rank 0 in the profiled pass that follows the timed region)",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_per_step": fam["gemm"][1] // args.steps, "avg_launch_ms": fam["gemm"][0] / max(fam["gemm"][1], 1),
                "traffic": args.gemm_traffic,
                "traffic_note": "dram bytes are not measurable inside a plain run: pass --gemm-traffic from the ncu capture of "
                                "this command (scripts/collect_profiles.sh -> profiles/)",
                "traffic_committed_capture": load_traffic() if args.workload == "so400m-384" else None,
                "share_of_rank0_busy_time": shares}
        by_type = pipe.engine.gemm_flops_by_type(my_images)
        roof["gemm_by_type"] = {k: {"achieved": by_type[k] / (fam_all[k][0] / 1e3) / 1e12, "frac": by_type[k] / (fam_all[k][0] / 1e3) / 1e12 / peak,
                                    "share_of_rank0_busy_time": fam_all[k][0] / busy_ms, "launches": fam_all[k][1]}
                                for k in by_type if fam_all[k][0] > 0}
        att_flops = 4.0 * arch.tokens ** 2 * arch.hidden_size * arch.num_hidden_layers * my_images
        if fam["attention"][0] > 0:
            a = att_flops / (fam["attention"][0] / 1e3) / 1e12
            roof["attention"] = {"kernel": "attention_dq_kernel", "achieved": a, "peak": peak, "unit": "TFLOP/s",
                                 "frac": a / peak, "avg_launch_ms": fam["attention"][0] / max(fam["attention"][1], 1)}
        # memory-bound kernels: algorithmic bytes per call (SURVEY.md §8d) / CUDA-event time, against the measured copy rate
        hb = float(peaks["hbm_gbs"])
        N, D, Kp = arch.tokens, arch.hidden_size, (3 * arch.patch_size ** 2 + 63) // 64 * 64
        for e in (hbm_entry("patchify_u8_rows_kernel", 3 * S * S + N * Kp * 2, my_images, *fam["patchify"], hb),
                  hbm_entry("map_attention_kernel", N * 2 * D * 2, my_images, *fam["map_attention"], hb),
                  hbm_entry("layernorm_bf16_kernel (post-LN of all tokens + the pooling head's LN)",
                            (N + 1) * D * 4, my_images, *fam["layernorm"], hb),
                  hbm_entry("gray256: luma + clahe_lut + clahe_apply + resample_rows + resample_cols",
                            3 * S * S + 256 * 256 * 4, my_images, *stages.get("gray256", (0, 0)), hb),
                  hbm_entry("freq_rows_kernel + freq_cols_kernel", 256 * 256 * 4 + 96, my_images, *stages.get("freq", (0, 0)), hb)):
            if e:
                hbm.append(e)
    line = {
        "metric": METRICS.get(args.workload, METRIC), "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {arch_name} detect (backbone+H-B head+gray256/CLAHE+freq features+G2 fusion+CORAL)",
                   "per_gpu_batch": B, "global_batch": B * world, "tokens": arch.tokens, "parallelism": f"dp{world}",
                   "sub_batch": sub, "schedule": "one call per step" if world == 1 else
                   f"work queue of {len(plan)} units ({sub}-image units, then a tail of {sub // 2}- and {sub // 4}-image ones) shared "
                   "by the ranks; one all-reduce(sum) of the zero-filled record slab (= all-gather under dynamic ownership) after "
                   "the last step",
                   "l2": f"per-step inputs ({B * S * S * 3 / 1e6:.0f} MB of u8 images) and activations are >> the 126 MB L2; no flush needed",
                   "weights": "random init (seeded), bf16", "fuse_ln": bool(args.fuse_ln),
                   "residual_stream": "two bf16 tensors (hi + lo)" if args.precise_residual else "bf16",
                   "cuda_graphs": bool(args.graphs)},
        "tensor_pipe_frac_of_step": arch.flops_per_image() * value / world / 1e12 / float(peaks["bf16_tflops_sustained"]),
        "clocks": {k: clocks.get(k) for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples")},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": dt_e2e / args.steps * 1e3, "api": "DetectionPipeline.detect_many (pinned host u8 in, numpy records out)"},
        "gpu_launches": int(launches // args.steps),
        "roofline": roof,
        "roofline_hbm": hbm,
        "per_rank": per_rank,
    }
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(args.workload)
        t1 = ref.run(1, seed=99)
        n = max(1, min(16, int(12.0 / max(t1, 1e-3))))
        t = ref.run(n, seed=5)
        line["cpu_baseline"] = {"value": n / t, "unit": "images/s", "cores": ref.cores, "kind": ref.kind,
                                "sample": ref.describe(n) + f"; one timed pass of {t:.1f} s after a 1-image warm-up"}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# Auxiliary workloads (BASELINE.json configs 4 and 5, and the small-batch latency a serving caller sees).  Not the driver's
# headline: each prints one JSON line with its own metric; numbers land in profiles/ via scripts/collect_profiles.sh.
# ---------------------------------------------------------------------------------------------------------
def _event_ms(fn, iters, warm=3):
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / iters


def run_latency(args):
    """Small-batch latency of the whole detection step (what detect_core issues per upload: 1 view, the 6 views of
    deepfake-detector-v2/app.py:1418-1430, the 9 crops of appv3.py:3315-3350), eager launches vs CUDA-graph replay."""
    import torch

    from dfd import _lib, pipeline, scoring, weights
    from dfd.engine import ARCHS

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {}
    for wl in ("base-224", "so400m-384"):
        arch = ARCHS[WORKLOADS[wl][0]]
        bsd = weights.random_vision_state_dict(arch, seed=0, device=dev)
        st = scoring.ScoringStack(dev, weights.random_freq_mlp_g2(2), weights.random_fusion_g2(3), [-1.0, -0.2, 0.3, 1.5], 1.0)
        pipe = pipeline.DetectionPipeline(arch, bsd, weights.random_classifier_head("B", arch.hidden_size, 1), st, device=0,
                                          max_batch=64, fuse_ln=True)
        del bsd
        S = arch.image_size
        for B in (1, 6, 9, 32):
            x = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, device=dev)
            row = {}
            for mode in ("eager", "graph"):
                pipe.engine.set_graphs(mode == "graph")
                r0 = pipe.engine.graph_replays
                ms = _event_ms(lambda: pipe.pack(pipe.detect_device(x, None, clahe=True)), iters=args.steps)
                row[mode + "_ms"] = ms
                if mode == "graph":
                    row["graph_replays"] = pipe.engine.graph_replays - r0
            row["images_per_s_graph"] = B / row["graph_ms"] * 1e3
            out[f"{wl}/B={B}"] = row
        pipe.engine.close()
        del pipe
    print(json.dumps({"metric": "detection step latency, small batches (u8 images resident in HBM -> score records on the device)",
                      "unit": "ms", "value": out["so400m-384/B=6"]["graph_ms"], "higher_is_better": False, "n_gpus": 1,
                      "steps": args.steps, "warmup": 3, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": "latency: 1 / 6 / 9 / 32 views per call, base-224 and so400m-384, eager vs CUDA graph"},
                      "gpu_launches": int(_lib.load().dfd_launch_count()), "table": out}), flush=True)


def run_cifake(args):
    """BASELINE config 4: 32x32 u8 images resampled to 224 inside the patch kernel (cifake_binary_classifier.py:714-749),
    base-patch16-224 backbone + head H-D, batch sweep."""
    import torch

    from dfd import _lib, cifake, dropin, weights
    from dfd.engine import ARCHS

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name = WORKLOADS["base-224"][0]
    model = dropin.FastBinaryClassifier("small", device=dev, arch=name, max_batch=1024,
                                        head_state=weights.random_fast_classifier_head("small", ARCHS[name].hidden_size))
    sweep = cifake.throughput_sweep(model, batches=(256, 512, 1024, 2048, 4096, 8192), side=32, iters=args.steps)
    best = max(sweep, key=sweep.get)
    arch = model.arch
    peaks = load_peaks()
    print(json.dumps({"metric": "images/sec CiFake 32->224 binary classifier (FastBinaryClassifier, base-patch16-224)",
                      "unit": "images/s", "value": sweep[best], "higher_is_better": True, "n_gpus": 1, "steps": args.steps,
                      "warmup": 1, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": "cifake: 32x32 u8 -> bilinear 224 in the patch kernel -> backbone -> head H-D",
                                 "best_batch": best, "engine_max_batch": 1024},
                      "tensor_pipe_frac": arch.flops_per_image() * sweep[best] / 1e12 / float(peaks["bf16_tflops_sustained"]),
                      "gpu_launches": int(_lib.load().dfd_launch_count()),
                      "sweep": {str(k): v for k, v in sweep.items()}}), flush=True)


def run_head_train(args):
    """BASELINE config 5: head-only training steps (train_fusion_head_only.py:406-453) on cached logits — fused forward/backward
    kernel, ONE all-reduce of the 196-float bucket over NCCL, clip + AdamW on every rank — and the FreqMLP trainer's step
    (6 495-float bucket).  Global batch 32 / 128 as in the reference scripts, sharded over the ranks."""
    import numpy as np
    import torch

    from dfd import _lib, distributed, train_freq, train_fusion

    rank, world, local = distributed.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    rng = np.random.default_rng(0)
    n = 32 * 64
    y = torch.from_numpy((rng.random(n) > 0.5).astype(np.float32))
    zs = torch.from_numpy((rng.normal(0, 2, n) + 2.0 * (y.numpy() - 0.5)).astype(np.float32))
    zf = torch.from_numpy((rng.normal(0, 2, n) + 1.0 * (y.numpy() - 0.5)).astype(np.float32))
    feats = torch.from_numpy((rng.normal(0.2, 0.7, (n, 24)) + 0.6 * (y.numpy()[:, None] - 0.5)).astype(np.float32))
    torch.manual_seed(11)
    t0 = time.perf_counter()
    train_fusion.fit_fusion_head(zf, zs, y, batch_size=32, epochs=1, device=dev, verbose=False)       # warm-up epoch
    torch.cuda.synchronize()
    epochs = args.steps
    t0 = time.perf_counter()
    train_fusion.fit_fusion_head(zf, zs, y, batch_size=32, epochs=epochs, device=dev, verbose=False)
    torch.cuda.synchronize()
    dt_fusion = time.perf_counter() - t0
    torch.manual_seed(5)
    train_freq.fit_freq_mlp(feats, y, epochs=1, batch_size=128, lr=1e-3, device=dev, dropout=0.0, verbose=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    train_freq.fit_freq_mlp(feats, y, epochs=epochs, batch_size=128, lr=1e-3, device=dev, dropout=0.0, verbose=False)
    torch.cuda.synchronize()
    dt_freq = time.perf_counter() - t0
    dt_fusion = distributed.max_over_ranks(dt_fusion, dev)
    dt_freq = distributed.max_over_ranks(dt_freq, dev)
    if rank == 0:
        steps_fusion, steps_freq = epochs * (n // 32), epochs * (n // 128)
        print(json.dumps({"metric": "head-only training steps/sec (fusion head, global batch 32, all-reduce of 196 floats)",
                          "unit": "steps/s", "value": steps_fusion / dt_fusion, "higher_is_better": True, "n_gpus": world,
                          "steps": steps_fusion, "warmup": n // 32, "dtype": "f32", "data": "synthetic", "scaling": "strong",
                          "config": {"workload": "head-train: fit_fusion_head + fit_freq_mlp on cached logits / features, "
                                                 "including the per-epoch evaluation pass, host loop timed by wall clock"},
                          "freq_mlp_steps_per_s": steps_freq / dt_freq, "freq_mlp_bucket_floats": 6495,
                          "us_per_fusion_step": dt_fusion / steps_fusion * 1e6, "us_per_freq_step": dt_freq / steps_freq * 1e6,
                          "gpu_launches": int(_lib.load().dfd_launch_count())}), flush=True)


def run_library(args):
    """The 'library' comparison point of SURVEY.md §8(d): the SAME HF model the reference calls (transformers.SiglipVisionModel,
    Siglip2sidafrozen.py:753,787) run eagerly by PyTorch on this B200 — bf16 autocast, SDPA attention, inference_mode, normalised
    fp32 NCHW input resident on the device.  None of this repository's kernels is on that path (gpu_launches = 0): the line says
    what stock PyTorch + cuBLAS + its attention library deliver on the hardware the product is measured on."""
    import torch
    from transformers import SiglipVisionConfig, SiglipVisionModel

    from dfd.engine import ARCHS

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peaks = load_peaks()
    table = {}
    for wl, B in (("so400m-384", args.batch or 64), ("base-224", args.batch or 256)):
        a = ARCHS[WORKLOADS[wl][0]]
        cfg = SiglipVisionConfig(hidden_size=a.hidden_size, intermediate_size=a.intermediate_size, num_hidden_layers=a.num_hidden_layers,
                                 num_attention_heads=a.num_attention_heads, image_size=a.image_size, patch_size=a.patch_size)
        cfg._attn_implementation = "sdpa"
        torch.manual_seed(0)
        m = SiglipVisionModel(cfg).to(dev).eval()
        x = torch.randint(0, 256, (B, a.image_size, a.image_size, 3), dtype=torch.uint8, device=dev)
        x = x.permute(0, 3, 1, 2).float().div_(255.0).mul_(2.0).sub_(1.0).contiguous()

        def step():
            with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
                return m(pixel_values=x).pooler_output

        ms = _event_ms(step, iters=args.steps, warm=max(args.warmup, 3))
        ips = B / ms * 1e3
        table[wl] = {"batch": B, "ms_per_step": ms, "images_per_s": ips,
                     "tensor_pipe_frac_of_sustained": a.flops_per_image() * ips / 1e12 / float(peaks["bf16_tflops_sustained"])}
        del m, x
        torch.cuda.empty_cache()
    print(json.dumps({"metric": "images/sec, backbone only, transformers.SiglipVisionModel eager on one B200 (library comparison point)",
                      "impl": "library", "unit": "images/s", "value": table["so400m-384"]["images_per_s"], "higher_is_better": True,
                      "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "dtype": "bf16 autocast", "data": "synthetic",
                      "config": {"workload": "library: HF SiglipVisionModel, bf16 autocast + SDPA, inference_mode, fp32 NCHW input on the device; "
                                             "so400m-384 and base-224"},
                      "gpu_launches": 0, "table": table}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 5; latency 20 calls per shape, cifake 3 calls per batch, head-train 3 epochs)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS) + ["latency", "cifake", "head-train", "library"], default="so400m-384",
                    help="so400m-384 (the driver's headline, BASELINE configs[2]) | base-224 (configs[1]) | latency | cifake "
                         "(configs[3]) | head-train (configs[4]) | library (stock PyTorch eager run of the HF model on the same GPU)")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: fix the GLOBAL batch (e.g. 512) and give every GPU global/N images per step; 0 = weak scaling")
    ap.add_argument("--max-batch", type=int, default=512, help="engine workspace batch (larger batches are chunked)")
    ap.add_argument("--sub-batch", type=int, default=0,
                    help="images per work-queue unit (default: the whole batch on one GPU, a quarter of it on several)")
    ap.add_argument("--gemm-traffic", type=float, default=None,
                    help="dram bytes per GEMM launch from an ncu --set full capture of this command, else null")
    ap.add_argument("--fuse-ln", type=int, default=1, help="1 = LayerNorm folded into the qkv/fc1 GEMMs")
    ap.add_argument("--graphs", type=int, default=1, help="1 = the engine forward is replayed as a CUDA graph (dfd_engine_set_graphs)")
    ap.add_argument("--precise-residual", type=int, default=0,
                    help="1 = two-bf16 residual stream (dfd_engine_set_precise_residual): the reference's fp32 residual "
                         "accumulation, a few percent slower; 0 = the default bf16 stream")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the score records of the last timed step to DIR/<field>.npy (float32), to compare two builds")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"latency": 20, "cifake": 3, "head-train": 3}.get(args.workload, 5)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs covers the so400m-384 and base-224 workloads of --impl ours")
    if args.impl == "reference":
        if args.workload not in WORKLOADS:
            raise SystemExit("--impl reference covers the so400m-384 and base-224 workloads")
        run_reference_arm(args)
    elif args.workload == "latency":
        run_latency(args)
    elif args.workload == "cifake":
        run_cifake(args)
    elif args.workload == "head-train":
        run_head_train(args)
    elif args.workload == "library":
        run_library(args)
    else:
        run_ours(args)
    try:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()

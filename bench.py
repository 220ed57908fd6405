#!/usr/bin/env python
"""Benchmark of the CaRA fine-tuning hot path on B200 (BASELINE.json: fine-tune images/sec, ViT-B/16 CaRA r16).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (the reference's CPU path, oracle port, host cores)

One "step" = one fine-tune iteration (reference vit_cp.py:45-50: forward, CE, backward, AdamW over CP*+head) on
a synthetic batch of 256 images per GPU (weak scaling; frozen backbone replicated, one NCCL all-reduce of the flat
CP+head gradient per step).  Prints ONE JSON line (rank 0).  --config selects the other BASELINE.json configurations
(vitl16_r32 / vith14_r32 / vitb16_eval); --global-batch G fixes the GLOBAL batch instead (strong scaling, configs[2]).
The CPU arm (--impl reference, and cpu_baseline in the default line) is BASELINE configs[0] exactly as BASELINE.md
section 5 specifies it: ViT-B/16 rank 8 fp32 batch 32, 1 warm-up + best of 3, oracle port, all host threads.
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy; model and batches are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[1] (the metric's configuration) and the larger data-parallel ones
    "vitb16_r16": dict(model="vit_base_patch16_224_in21k", embed_dim=768, depth=12, num_heads=12, patch=16, rank=16,
                       batch=256, gflop_per_image=74.24),
    "vitl16_r32": dict(model="vit_large_patch16_224_in21k", embed_dim=1024, depth=24, num_heads=16, patch=16, rank=32,
                       batch=256, gflop_per_image=264.60),
    "vith14_r32": dict(model="vit_huge_patch14_224_in21k", embed_dim=1280, depth=32, num_heads=16, patch=14, rank=32,
                       batch=128, gflop_per_image=711.95),
    # BASELINE.json configs[4]: --evaluate mode, CP delta merged into the frozen weights, inference batch 1024
    "vitb16_eval": dict(model="vit_base_patch16_224_in21k", embed_dim=768, depth=12, num_heads=12, patch=16, rank=16,
                        batch=1024, gflop_per_image=35.13, eval=True),
}
NUM_CLASSES = 100
METRIC = "fine-tune images/sec, ViT-B/16 CaRA r16, 1/2/4/8 B200; fused GEMM % TC peak"
METRICS = {"vitb16_r16": METRIC,
           "vitl16_r32": "fine-tune images/sec, ViT-L/16 CaRA r32 data-parallel (BASELINE configs[2])",
           "vith14_r32": "fine-tune images/sec, ViT-H/14 CaRA r32 data-parallel, 257 tokens (BASELINE configs[3])"}
WORKLOADS = {
    "vitb16_r16": "ViT-B/16 CaRA rank=16 bf16 fine-tune step (fwd + CE + dX-only bwd + factor grads + AdamW over "
                  "CP*+head), batch 256 per GPU, 224x224, 100 classes, random-init weights",
    "vitl16_r32": "ViT-L/16 CaRA rank=32 bf16 data-parallel fine-tune step, 224x224, 100 classes, random-init weights",
    "vith14_r32": "ViT-H/14 CaRA rank=32 bf16 data-parallel fine-tune step, 224x224 (257 tokens), 100 classes, "
                  "random-init weights"}


def gemm_traffic(config_key):
    """DRAM bytes per gemm_cp_kernel launch (launch-weighted over one step) from the committed ncu --set full
    captures (profiles/r01_traffic.json); None when no capture exists for this configuration."""
    import glob
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        d = json.load(open(p))
        if d.get("config_key") == config_key:
            return float(d["avg_dram_bytes_per_launch"])
    return None


def gemm_ncu(config_key):
    """Second denominator for the GEMM roofline: ncu's sm__pipe_tensor_cycles_active, time-weighted over the
    fused-projection shapes of one step, from the newest committed capture (profiles/rNN_traffic.json)."""
    import glob
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        d = json.load(open(p))
        if d.get("config_key") == config_key and "tensor_pipe_pct_time_weighted" in d:
            return {"tensor_pipe_pct_time_weighted": d["tensor_pipe_pct_time_weighted"], "source": os.path.basename(p)}
    return {}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["bf16_tflops_sustained"]), float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi SM clock / throttle-reason samples taken DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        pw = sorted(v for v in (num(r[6]) for r in self.rows if len(r) >= 8) if v is not None)
        pl = [v for v in (num(r[7]) for r in self.rows if len(r) >= 8) if v is not None]
        # board power under load next to its limit: with sw_power_cap active the step is bounded by energy, not by the
        # sum of its kernels' isolated times (DESIGN.md section 6)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": reasons, "samples": len(sm)}
        if len(pw) >= 15:      # nvidia-smi's power.draw is a ~1 s running average: only meaningful over a window of seconds
            out.update({"power_w": pw[len(pw) // 2], "power_limit_w": max(pl) if pl else None})
        return out


def build_model(cfg, device):
    import torch
    from cara_b200 import train as T
    from cara_b200.vit import create_model
    from oracle_free_init import init_synthetic  # noqa: F401  (defined below, injected into sys.modules)
    from src.cara.cara import cara
    torch.manual_seed(0)
    vit = create_model(cfg["model"], drop_path_rate=0.1)
    vit = cara({"model": vit, "rank": cfg["rank"], "scale": 1.0, "l_mu": 1.0, "l_std": 0.1})
    vit.reset_classifier(NUM_CLASSES)
    init_synthetic(vit, cfg["rank"])
    vit = vit.to(device)
    trainable = T.freeze_backbone(vit)
    opt = T.FusedAdamW(T.FlatTrainable(trainable), lr=1e-3, weight_decay=1e-4)
    vit.train()
    return vit, opt


def apply_weight_dropout(vit, mode):
    from cara_b200 import wdrop
    wdrop.set_weight_dropout(vit, mode)


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(loss, opt):
    """What a fine-tune step leaves its caller, copied to the host: the loss it returns and every trainable tensor (CP
    factors and head) after its AdamW update.  Gradients are left out: AdamW's first updates move each element by about
    lr * sign(g), so elements whose gradient is rounding noise (fp32 atomics) go either way.  Two runs of the default
    configuration with --steps 20 --warmup 5 on one B200 (1,000 W limit) differed in the last gradient by up to 3e-1
    relative, in the parameters by at most 1.3e-2 relative and in the loss by 8e-3."""
    flat = opt.flat.flat.detach().cpu().numpy()
    out = {"loss": loss.detach().float().cpu().numpy().reshape(1)}
    for n, p in opt.flat.named:
        a, b = opt.flat.slices[n]
        out["param." + n] = flat[a:b].reshape(p.shape)
    return out


def dump_outputs(directory, arrays):
    """--dump-outputs: one float32 / float64 DIR/<name>.npy per array."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(directory, name + ".npy"), a)


def _install_init_module():
    """Random-init weights of the architecture + non-default CP factors (the reference's default init makes every
    delta exactly zero, cara.py:128,132; SURVEY D.3 recipe keeps the adapter numerically alive)."""
    import types

    import torch

    def init_synthetic(vit, rank):
        g = torch.Generator().manual_seed(1234)
        sa, sp = (0.01 / rank ** 0.5) ** 0.25, (0.01 / rank ** 0.5) ** (1.0 / 3.0)
        with torch.no_grad():
            for n, p in vit.named_parameters():
                if n.startswith("CP_A"):
                    p.copy_(torch.randn(p.shape, generator=g) * sa)
                elif n.startswith("CP_P"):
                    p.copy_(torch.randn(p.shape, generator=g) * sp)
                elif n.startswith("CP_bias"):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.02)
                elif n.endswith(".bias"):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    mod = types.ModuleType("oracle_free_init")
    mod.init_synthetic = init_synthetic
    sys.modules["oracle_free_init"] = mod


def run_cuda(args):
    import torch
    import torch.distributed as dist
    from cara_b200 import kernels as K
    from cara_b200 import train as T

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if args.gpus > 1 and world == 1:
            raise SystemExit("bench.py --gpus %d must be launched with torchrun (one rank per GPU)" % args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _install_init_module()
    cfg = CONFIGS[args.config]
    B = args.batch or cfg["batch"]
    strong = args.global_batch > 0
    if strong:                                   # strong scaling (BASELINE configs[2]): the GLOBAL batch is fixed
        if args.global_batch % world != 0:
            raise SystemExit("--global-batch must be divisible by the number of GPUs")
        B = args.global_batch // world
        if args.accum == 0:                      # activations are kept for one micro-batch of the config's batch size
            args.accum = max(1, B // cfg["batch"])
    if args.accum == 0:
        args.accum = 1
    vit, opt = build_model(cfg, dev)
    apply_weight_dropout(vit, args.weight_dropout)
    if cfg.get("eval"):
        return run_eval(args, cfg, vit, dev, world, rank)
    img = 224
    g = torch.Generator().manual_seed(4321 + rank)
    host_x = [torch.randn(B, 3, img, img, generator=g).pin_memory() for _ in range(2)]
    host_y = [torch.randint(0, NUM_CLASSES, (B,), generator=g).pin_memory() for _ in range(2)]
    dev_x = [t.to(dev) for t in host_x]
    dev_y = [t.to(dev) for t in host_y]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------------------ device-resident throughput ("value")
    # zero_grad + forward + CE + backward are replayed from one CUDA graph (cara_b200.train.GraphedStep); the
    # all-reduce and the fused AdamW kernel are launched eagerly after each replay.
    if args.accum < 1 or B % args.accum != 0 or (args.no_graph and args.accum != 1):
        raise SystemExit("--accum must divide the per-GPU batch (and needs the CUDA-graph step)")
    if args.no_graph:
        step = lambda x, y: T.train_step(vit, opt, x, y, world)          # noqa: E731
    else:
        step = T.GraphedStep(vit, opt, dev_x[0][:B // args.accum], dev_y[0][:B // args.accum], world, accumulate=args.accum)
    for i in range(args.warmup):
        step(dev_x[i % 2], dev_y[i % 2])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = K.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        loss = step(dev_x[i % 2], dev_y[i % 2])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = K.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    loss_value = float(loss)
    # taken now: the roofline and end-to-end passes below keep training the same model
    outputs = step_outputs(loss, opt) if args.dump_outputs and rank == 0 else None

    # ------------------------------------------------------------ roofline of the dominant kernel: the same step run
    # eagerly with CUDA events around every fused-projection launch (events inside a replayed graph cannot be timed)
    K.gemm_events = []
    mb = B // args.accum                                      # (one micro-batch when gradients are accumulated)
    for i in range(2):
        T.train_step(vit, opt, dev_x[i % 2][:mb], dev_y[i % 2][:mb], world)
    torch.cuda.synchronize()
    gemm_events, K.gemm_events = K.gemm_events, None
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in gemm_events)
    gemm_flops = sum(f for _, _, f in gemm_events)

    # ------------------------------------------------------------ end-to-end: host buffers, H2D + D2H in the timed region
    copy_stream = torch.cuda.Stream(device=dev)
    stage_x = [torch.empty_like(dev_x[0]) for _ in range(2)]
    stage_y = [torch.empty_like(dev_y[0]) for _ in range(2)]
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[s])            # the step that last used this slot has finished
            stage_x[s].copy_(host_x[s], non_blocking=True)
            stage_y[s].copy_(host_y[s], non_blocking=True)
            ready[s].record(copy_stream)

    def e2e_loop(n):
        losses = []
        prefetch(0)
        for i in range(n):
            s = i % 2
            if i + 1 < n:
                prefetch(i + 1)
            torch.cuda.current_stream().wait_event(ready[s])
            l = step(stage_x[s], stage_y[s])
            loss_host[s].copy_(l.detach(), non_blocking=True)     # D2H read of this step's loss
            done[s].record()                                       # (graph mode: stage -> static copy has been enqueued)
            ev = torch.cuda.Event(); ev.record()
            losses.append((ev, s))
            if i > 0:                                            # consume the previous step's loss on the host
                pe, ps = losses[i - 1]
                pe.synchronize()
                _ = float(loss_host[ps])
        losses[-1][0].synchronize()
        return float(loss_host[losses[-1][1]])

    e2e_loop(2)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    e2e_loop(args.steps)
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)

    if world > 1:
        t = torch.tensor([ms, ms_e2e, gemm_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, gemm_ms = [float(v) for v in t]
    total_images = B * world * args.steps
    peak_tf, peak_hbm, peak_src = peaks()
    ncu = gemm_ncu(args.config)
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    out = {
        "metric": METRICS[args.config], "value": total_images / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config],
                   "config_key": args.config, "batch_per_gpu": B, "global_batch": B * world,
                   "tokens": (224 // cfg["patch"]) ** 2 + 1,
                   "parallelism": "dp%d" % world, "l2": "per-step working set (>10 GB of activations) exceeds the 126 MB L2",
                   "drop_path": 0.1,
                   "weight_dropout": "not applied (documented deviation; --weight-dropout exact selects the slow path)"
                   if args.weight_dropout == "skip" else "exact (reference semantics: 3 GEMMs per projection)",
                   "cuda_graph": not args.no_graph, "micro_batches": args.accum,
                   "update_in_graph": bool(getattr(step, "capture_update", False)),
                   "algorithmic_gflop_per_image": cfg["gflop_per_image"]},
        "e2e": {"value": total_images / (ms_e2e * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": int(host_x[0].numel() * 4 + host_y[0].numel() * 8), "d2h_bytes_per_step": 4,
                "note": "pinned host batches, copy stream prefetch, loss read back every step"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_cp_kernel (fused CP projections fwd + dX, %d launches over 2 eagerly enqueued steps)" % len(gemm_events),
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": gemm_traffic(args.config), "traffic_unit": "DRAM bytes per launch (ncu --set full, newest profiles/rNN_traffic.json)",
                     "algorithmic_flops_per_launch": gemm_flops / max(1, len(gemm_events)),
                     "peak_source": peak_src,
                     "timing": "CUDA events around each launch of two eagerly enqueued steps right after the timed loop "
                               "(nodes of a replayed graph cannot be timed individually)",
                     "ncu_tensor_pipe_pct": ncu.get("tensor_pipe_pct_time_weighted"),
                     "ncu_source": ncu.get("source"),
                     "step_frac_of_peak": cfg["gflop_per_image"] * 1e9 * B / (ms / args.steps * 1e-3) / 1e12 / peak_tf},
        "loss": loss_value,
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_reference(args, steps=3, warmup=1)
        print(json.dumps(out), flush=True)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        if hasattr(step, "release"):
            step.release()                       # captured collectives must be gone before the communicator is
        dist.barrier()
        dist.destroy_process_group()


def run_eval(args, cfg, vit, dev, world, rank):
    """--evaluate path (vit_cp.py:168-173, :73-82): merge the CP delta into the frozen weights once
    (cara_b200.merge.merge_cara), then time plain forwards + arg-max at the config's inference batch."""
    import torch
    import torch.distributed as dist
    from cara_b200 import kernels as K
    from cara_b200.merge import merge_cara
    B = args.batch or cfg["batch"]
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    merged = merge_cara(vit)                     # first call: module loading, allocator growth
    torch.cuda.synchronize()
    t0.record()
    merged = merge_cara(vit)                     # timed: 4 x depth reconstruction-kernel launches + their staging
    t1.record()
    torch.cuda.synchronize()
    merge_ms = t0.elapsed_time(t1)
    g = torch.Generator().manual_seed(4321 + rank)
    host_x = [torch.randn(B, 3, 224, 224, generator=g).pin_memory() for _ in range(2)]
    dev_x = [t.to(dev) for t in host_x]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def fwd(x):
        with torch.no_grad():
            return vit(x).argmax(1)

    for i in range(args.warmup):
        fwd(dev_x[i % 2])
    barrier()
    launches0 = K.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        pred = fwd(dev_x[i % 2])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = K.launch_count - launches0
    # the predicted classes of the last timed batch (float64 holds every class index exactly)
    outputs = {"pred": pred.double().cpu().numpy()} if args.dump_outputs and rank == 0 else None
    stage = [torch.empty_like(dev_x[0]) for _ in range(2)]
    pred_host = torch.zeros(B, dtype=torch.int64).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):                               # H2D of batch i on the copy stream, overlapping forward i-1
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[s])
            stage[s].copy_(host_x[s], non_blocking=True)
            ready[s].record(copy_stream)

    t0.record()
    prefetch(0)
    for i in range(args.steps):
        s = i % 2
        if i + 1 < args.steps:
            prefetch(i + 1)
        torch.cuda.current_stream().wait_event(ready[s])
        pred_host.copy_(fwd(stage[s]), non_blocking=True)
        done[s].record()
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = [float(v) for v in t]
    peak_tf, _, peak_src = peaks()
    total = B * world * args.steps
    out = {"metric": "eval images/sec, ViT-B/16 CaRA r16 merged (--evaluate)", "value": total / (ms * 1e-3), "unit": "images/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "ViT-B/16 --evaluate forward, CP delta merged into the frozen weights by the reconstruction "
                                  "kernel, inference batch %d per GPU" % B, "config_key": args.config,
                      "merged_projections": merged, "merge_ms": merge_ms,
                      "algorithmic_gflop_per_image": cfg["gflop_per_image"]},
           "e2e": {"value": total / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": int(host_x[0].numel() * 4),
                   "d2h_bytes_per_step": B * 8},
           "gpu_launches": launches,
           "roofline": {"bound": "tensor", "kernel": "whole eval forward vs dense bf16 peak",
                        "achieved": cfg["gflop_per_image"] * 1e9 * B / (ms / args.steps * 1e-3) / 1e12, "peak": peak_tf,
                        "unit": "TFLOP/s", "frac": cfg["gflop_per_image"] * 1e9 * B / (ms / args.steps * 1e-3) / 1e12 / peak_tf,
                        "traffic": None, "peak_source": peak_src}}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


CPU_CONFIG = dict(embed_dim=768, depth=12, num_heads=12, patch=16, rank=8, batch=32)   # BASELINE.json configs[0]
CPU_WORKLOAD = ("BASELINE configs[0]: ViT-B/16 CaRA rank=8 fp32 fwd+bwd+AdamW step on the host CPU, batch 32 synthetic "
                "224x224, 100 classes, random-init weights, train mode as shipped (weight dropout 0.1, DropPath 0.1)")


def cpu_reference(args, steps=3, warmup=1):
    """The reference's CPU path at BASELINE config 1 exactly as BASELINE.md section 5 / SURVEY 8(d) specify it: the
    loop body of vit_cp.py:45-50 (forward, CE, backward through the materialised deltas, AdamW(lr 1e-3, wd 1e-4) over
    CP* + head) in train mode as shipped, ViT-B/16, rank 8, fp32, batch 32, all host threads, ``warmup`` untimed steps
    then best of ``steps``.  The reference is pure Python on timm/tensorly, which are not in this image, so what runs
    is the oracle port (oracle/cara_oracle.py, pinned to the reference's own outputs by tests/test_oracle_golden.py):
    ``kind`` says "port".  Returns the steps / warm-ups actually executed."""
    import torch
    from oracle import cara_oracle as O
    c = dict(CPU_CONFIG)
    c["rank"] = args.cpu_rank or c["rank"]
    c["batch"] = args.cpu_batch or c["batch"]
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = O.Geometry(embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"], patch=c["patch"],
                   num_classes=NUM_CLASSES, rank=c["rank"])
    st = O.synthetic_state(g)
    x, y = O.synthetic_batch(g, c["batch"])
    opt = {}
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.train_step(st, opt, i + 1, g, x, y, 1.0, train=True, wdrop=0.1, drop_path=0.1)
        times.append(time.perf_counter() - t0)
    timed = times[warmup:]
    best = min(timed)
    return {"value": c["batch"] / best, "unit": "images/s", "cores": threads, "torch_threads": torch.get_num_threads(),
            "kind": "port",
            "sample": "%d timed steps (best of, after %d warm-up) of the ViT-B/16 rank-%d fp32 train step at batch %d "
                      "(BASELINE configs[0]) on the host CPU: oracle/cara_oracle.py = materialised deltas + weight "
                      "dropout + autograd + AdamW as the reference's vit_cp.py:45-50"
                      % (steps, warmup, c["rank"], c["batch"]),
            "sec_per_step": best, "sec_per_step_mean": sum(timed) / len(timed), "steps": steps, "warmup": warmup,
            "rank": c["rank"], "batch": c["batch"]}


def run_reference(args):
    """bench.py --impl reference: the CPU arm.  Always 1 warm-up + best of 3 (BASELINE.md section 5), whatever
    --steps / --warmup ask for -- and the line reports the counts that were actually executed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = cpu_reference(args, steps=3, warmup=1)
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "images/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": base["steps"], "warmup": base["warmup"],
           "steps_requested": args.steps, "warmup_requested": args.warmup,
           "ms_per_step": base["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": CPU_WORKLOAD, "config_key": "vitb16_r%d_cpu" % base["rank"],
                      "batch": base["batch"], "gpu_arm_config_key": args.config},
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cara_b200", choices=["cara_b200", "reference"])
    ap.add_argument("--config", default="vitb16_r16", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the config's)")
    ap.add_argument("--cpu-batch", type=int, default=0, help="batch of the CPU baseline (default: BASELINE configs[0], 32)")
    ap.add_argument("--cpu-rank", type=int, default=0, help="CP rank of the CPU baseline (default: BASELINE configs[0], 8)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--weight-dropout", default="skip", choices=["skip", "exact"],
                    help="exact: the reference's nn.Dropout(0.1) on the materialised delta weights (slow path)")
    ap.add_argument("--accum", type=int, default=0,
                    help="micro-batches per optimizer step (the per-GPU batch is split; activations kept for one); "
                         "default 1, or per-GPU batch / config batch with --global-batch")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: fix the GLOBAL batch (BASELINE configs[2]: 2048) and split it over the GPUs")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Kernel and step times of the key-tiled D = 80 attention (csrc/attention_tiled.cu, ViT-H/14 above 224 px), written as
one JSON file (default profiles/r05_attn_d80.json) with the card's name, power limit and the SM clock sampled while it
measured.

  * kernel times: CUDA events around each forward / backward pass, the 126 MB L2 overwritten (256 MB memset) before
    every pass; median over the passes.  The tiled backward includes its delta pre-pass (three launches); the
    whole-head backward includes its in-kernel delta pass.  Rates: algorithmic TFLOP/s (forward 4 N^2 D, backward
    10 N^2 D per head; the dQ kernel's recompute of S and dP is not counted).
  * A/B: whole-head (attention.cu) against tiled at (32, 257, 16) both directions and at (32, 401, 16) forward, in one
    process, alternating A/B over several rounds.
  * step: graph-replayed ViT-H/14 r32 train step (train.GraphedStep, bench.py's init) at 336 px, batch 64.  The share of
    the step spent in attention is the attention kernels' time over all kernels' time in a separate, profiled eager step
    (torch.profiler, CUDA activities).
"""
import argparse
import json
import os
import re
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

D = 80
BF16 = torch.bfloat16


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_" + q.replace(",", "|"): out[0] if out else None}


_flush = []


def timed(fn, reps):
    """Median device time (ms) of fn over ``reps`` passes, each after overwriting L2."""
    if not _flush:
        _flush.append(torch.empty(256 << 20, dtype=torch.uint8, device="cuda"))
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        _flush[0].zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def _inputs(B, N, H):
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(B * N * 3 * H * D, device="cuda", generator=g).to(BF16)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
    return qkv, d_o


def case(B, N, H, reps, path, backward=True):
    """path "tiled" or "whole_head"; forward (and backward) median ms and TFLOP/s."""
    from cara_b200 import kernels as K
    fwd, bwd = (K.attn_tiled_fwd, K.attn_tiled_bwd) if path == "tiled" else (K.attn_fwd, K.attn_bwd)
    qkv, d_o = _inputs(B, N, H)
    scale = D ** -0.5
    o, o_lo, lse = fwd(qkv, B, N, H, D, scale)
    heads = B * H
    t_f = timed(lambda: fwd(qkv, B, N, H, D, scale), reps)
    out = {"B": B, "N": N, "H": H, "path": path, "fwd_ms": round(t_f, 4),
           "fwd_tflops": round(4.0 * N * N * D * heads / t_f * 1e-9, 1)}
    if backward:
        t_b = timed(lambda: bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, scale), reps)
        out.update({"bwd_ms": round(t_b, 4), "bwd_tflops": round(10.0 * N * N * D * heads / t_b * 1e-9, 1)})
    return out


def ab(B, N, H, reps, rounds, backward):
    runs = []
    for _ in range(rounds):
        runs.append(case(B, N, H, reps, "whole_head", backward))
        runs.append(case(B, N, H, reps, "tiled", backward))
    keys = ["fwd_ms"] + (["bwd_ms"] if backward else [])
    med = {}
    for path in ("whole_head", "tiled"):
        for k in keys:
            v = sorted(r[k] for r in runs if r["path"] == path)
            med["%s_%s_median" % (path, k)] = v[len(v) // 2]
    for k in keys:
        med["tiled_over_whole_head_" + k] = round(med["tiled_%s_median" % k] / med["whole_head_%s_median" % k], 3)
    return {"B": B, "N": N, "H": H, "runs": runs, **med}


def vith14_336(batch):
    import bench
    from cara_b200 import train as T
    from cara_b200.vit import create_model
    from src.cara.cara import cara
    bench._install_init_module()
    from oracle_free_init import init_synthetic
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    vit = create_model("vit_huge_patch14_224_in21k", drop_path_rate=0.1, img_size=336)
    vit = cara({"model": vit, "rank": 32, "scale": 1.0, "l_mu": 1.0, "l_std": 0.1})
    vit.reset_classifier(bench.NUM_CLASSES)
    init_synthetic(vit, 32)
    vit = vit.to(dev)
    opt = T.FusedAdamW(T.FlatTrainable(T.freeze_backbone(vit)), lr=1e-3, weight_decay=1e-4)
    vit.train()
    x = torch.randn(batch, 3, 336, 336, device=dev)
    y = torch.randint(0, bench.NUM_CLASSES, (batch,), device=dev)
    return vit, opt, x, y


def step(batch, n_steps, rounds):
    from torch.profiler import ProfilerActivity, profile

    import bench
    from cara_b200 import train as T
    vit, opt, x, y = vith14_336(batch)
    graphed = T.GraphedStep(vit, opt, x, y)
    for _ in range(3):
        graphed(x, y)
    torch.cuda.synchronize()
    sampler = bench.ClockSampler(0)
    sampler.start()
    ms = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_steps):
            graphed(x, y)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / n_steps)
    clocks = sampler.stop()
    del graphed
    # kernel-time share of attention in one eager step (profiled separately: tracing slows the host, not the kernels)
    T.train_step(vit, opt, x, y, 1)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        T.train_step(vit, opt, x, y, 1)
        torch.cuda.synchronize()
    per = {ev.key: ev.device_time_total for ev in prof.key_averages() if ev.device_time_total > 0}
    total = sum(per.values())
    attn = {k: v for k, v in per.items() if re.search(r"attn_\w+", k)}
    v = sorted(ms)
    med = v[len(v) // 2]
    out = {"model": "vit_huge_patch14_224_in21k", "img": 336, "tokens": 577, "rank": 32, "batch": batch,
           "step_ms_median": round(med, 3), "step_ms_rounds": [round(t, 3) for t in ms],
           "img_per_s": round(batch / med * 1e3, 1),
           "eager_kernel_us_total": round(total, 1),
           "eager_attention_kernel_us": {re.search(r"attn_\w+", k).group(0): round(t, 1) for k, t in sorted(attn.items())},
           "attention_share_of_kernel_time": round(sum(attn.values()) / total, 4) if total else None,
           "clocks": clocks}
    del vit, opt
    torch.cuda.empty_cache()
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_attn_d80.json"))
    p.add_argument("--reps", type=int, default=20, help="timed passes per kernel case")
    p.add_argument("--rounds", type=int, default=3, help="A/B alternation rounds and step rounds")
    p.add_argument("--steps", type=int, default=10, help="graph replays per step round")
    p.add_argument("--batch", type=int, default=64)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attn_d80_time.py measures on the GPU; no CUDA device found")
    import bench
    res = {"card": card(), "l2": "overwritten (256 MB memset) before every timed kernel pass", "reps": a.reps,
           "rounds": a.rounds, "flops": "forward 4 N^2 D, backward 10 N^2 D per head (dQ recompute not counted)"}
    sampler = bench.ClockSampler(0)
    sampler.start()
    res["tiled"] = [case(B, N, H, a.reps, "tiled") for B, N, H in [(32, 577, 16), (16, 1025, 16)]]
    res["ab_n257"] = ab(32, 257, 16, a.reps, a.rounds, backward=True)
    res["ab_n401_fwd"] = ab(32, 401, 16, a.reps, a.rounds, backward=False)
    res["kernel_clocks"] = sampler.stop()
    res["step"] = step(a.batch, a.steps, a.rounds)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Kernel times of the key-tiled tcgen05 attention (csrc/attention_long.cu, D = 64, N > 256) and the train step above
224 px, written as one JSON file (default profiles/r03_attn_long.json) with the card's name and power limit.

  * kernel times: CUDA events around each forward / backward pass, the 126 MB L2 overwritten (256 MB memset) before
    every pass; median over the passes.  Backward = the two kernels fed with a precomputed delta, as in the train
    step, where the output projection's dX GEMM writes delta (EPI_DELTA).
  * rates: algorithmic TFLOP/s as DESIGN section 5 counts them (forward 4 N^2 D, backward 10 N^2 D per head; the dQ
    kernel's recompute of S and dP is not counted) and scores (N^2 per head) per second, next to the N = 197 kernels.
  * A/B at (64, 12, 401), where both paths run: the mma.sync kernels (a subprocess with CARA_ATTN_TC=0) against the
    new kernels, alternating A/B/A/B; both backward sides include their rowsum(dO (.) O) pass.
  * step: graph-replayed ViT-B/16 r16 train step (train.GraphedStep) at 384 px with batch 64 and 87 (87 x 577 tokens
    ~ 256 x 197) and at 224 px with batch 256.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

D = 64
BF16 = torch.bfloat16


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out[0] if out else None}


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


def attn_case(B, N, H, reps, precomputed_delta=True):
    from cara_b200 import kernels as K
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(B * N * 3 * H * D, device="cuda", generator=g).to(BF16)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
    scale = D ** -0.5
    o, o_lo, lse = K.attn_fwd(qkv, B, N, H, D, scale)
    t_f = timed(lambda: K.attn_fwd(qkv, B, N, H, D, scale), reps)
    if precomputed_delta:
        delta = (d_o.float() * (o.float() + o_lo.float())).view(B, N, H, D).sum(-1).permute(0, 2, 1).contiguous()
        t_b = timed(lambda: K.attn_bwd(qkv, None, None, lse, d_o, B, N, H, D, scale, delta=delta), reps)
    else:
        t_b = timed(lambda: K.attn_bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, scale), reps)
    heads = B * H
    return {"B": B, "N": N, "H": H, "fwd_ms": t_f, "bwd_ms": t_b,
            "fwd_tflops": 4.0 * N * N * D * heads / t_f * 1e-9, "bwd_tflops": 10.0 * N * N * D * heads / t_b * 1e-9,
            "fwd_gscores_per_s": float(N) * N * heads / t_f * 1e-6, "bwd_gscores_per_s": float(N) * N * heads / t_b * 1e-6}


def step_time(img, batch, steps=20):
    import bench
    from cara_b200 import train as T
    dev = torch.device("cuda", 0)
    bench._install_init_module()
    model = "vit_base_patch16_384" if img == 384 else "vit_base_patch16_224_in21k"
    vit, opt = bench.build_model(dict(model=model, rank=16), dev)
    x = torch.randn(batch, 3, img, img, device=dev)
    y = torch.randint(0, bench.NUM_CLASSES, (batch,), device=dev)
    step = T.GraphedStep(vit, opt, x, y)
    for _ in range(3):
        step(x, y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(x, y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    tokens = batch * ((img // 16) ** 2 + 1)
    del step, vit, opt
    torch.cuda.empty_cache()
    return {"img": img, "batch": batch, "tokens": tokens, "step_ms": ms, "img_per_s": batch / ms * 1e3}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_attn_long.json"))
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--ab-side", default=None, help=argparse.SUPPRESS)    # child of the A/B: print one case as JSON
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attn_long_time.py measures on the GPU; no CUDA device found")
    if a.ab_side is not None:
        print(json.dumps(attn_case(64, 401, 12, a.reps, precomputed_delta=False)))
        return
    res = {"card": card(), "l2": "overwritten (256 MB memset) before every timed pass", "reps": a.reps,
           "flops": "forward 4 N^2 D, backward 10 N^2 D per head (dQ recompute not counted)"}
    res["long"] = [attn_case(B, N, H, a.reps) for B, N, H in [(64, 577, 12), (32, 577, 16), (16, 1025, 12)]]
    res["short_n197"] = [attn_case(256, 197, 12, a.reps)]
    ab = []
    for _ in range(2):
        env = dict(os.environ, CARA_ATTN_TC="0")
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab-side=mma_sync", "--reps=%d" % a.reps],
                             env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
        ab.append(dict(json.loads(out), path="mma.sync (CARA_ATTN_TC=0)"))
        ab.append(dict(attn_case(64, 401, 12, a.reps, precomputed_delta=False), path="tcgen05 key-tiled"))
    res["ab_n401"] = ab
    res["step"] = [step_time(384, 64), step_time(384, 87), step_time(224, 256)]
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

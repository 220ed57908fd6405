#!/usr/bin/env python
"""What the CaRA rank costs on the bf16 path: the ViT-B/16 train step at ranks 16 / 32 / 64 and the rank-R skinny
kernels at Rp = 32 against Rp = 64, written as one JSON file (default profiles/r04_rank64.json) with the card's name,
power limit and SM clock from the same run.

  * step: graph-replayed ViT-B/16 train step (train.GraphedStep, bench.py's model and init), batch 256, 224 px.  The
    three ranks are built once and timed in turn, rank after rank, over several rounds; per rank the median of the
    rounds.  The SM clock and board power are sampled with nvidia-smi during the timed steps.
  * kernels at M = 50,432 (ViT-B/16, batch 256): rows forward (K = 768, one slice), rows backward (1 / 3 / 4 slices of
    768 columns), cols (Kc = 768 / 2304 / 3072 with 1 / 3 / 4 slices, column sums on).  CUDA events around each pass,
    the 126 MB L2 overwritten (256 MB memset) before every pass, median over the passes; Rp = 32 and Rp = 64 alternate.
    GB/s = bytes computed from the shapes (below) over the median time.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BF16 = torch.bfloat16
M = 50432
BYTES = {"rows_fwd": "X read once (2 M K) + T written (4 M Rp) + Uhat written (6 M Rp)",
         "rows_bwd": "G read once (2 M N) + T read (4 M Rp) + dThat written (6 M Rp)",
         "cols": "X read once (2 M Kc) + the hi and lo blocks of V read (4 M Rp per slice)"}


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


def kernel_cases(Rp):
    """(name, shape dict, bytes, callable) for one padded rank."""
    from cara_b200 import kernels as K
    g = torch.Generator(device="cuda").manual_seed(Rp)
    bf = lambda *s: (torch.randn(*s, device="cuda", generator=g) * 0.1).to(BF16)   # noqa: E731
    cases = []
    x = bf(M, 768)
    a_t2 = bf(2 * Rp, 768)
    sc1 = torch.randn(1, Rp, device="cuda", generator=g)
    cases.append(("rows_fwd", dict(K=768, S=1), 2 * M * 768 + 10 * M * Rp, lambda: K.adapter_rows_fwd(x, a_t2, sc1)))
    T = torch.randn(M, Rp, device="cuda", generator=g)
    for S in (1, 3, 4):
        G = bf(M, S * 768)
        b_t2 = bf(2 * Rp, 768)
        sc = torch.randn(S, Rp, device="cuda", generator=g)
        dsc = torch.zeros(S, Rp, device="cuda")
        cases.append(("rows_bwd", dict(N=S * 768, S=S), 2 * M * S * 768 + 10 * M * Rp,
                      lambda G=G, b_t2=b_t2, sc=sc, dsc=dsc: K.adapter_rows_bwd(G, b_t2, sc, T, dsc=dsc)))
    for Kc, S in ((768, 1), (2304, 3), (3072, 4)):
        X = bf(M, Kc)
        V = bf(M, S * 3 * Rp)
        out = torch.zeros(Kc // S, Rp, device="cuda")
        cs = torch.zeros(Kc, device="cuda")
        cases.append(("cols", dict(Kc=Kc, S=S), 2 * M * Kc + 4 * M * Rp * S,
                      lambda X=X, V=V, S=S, out=out, cs=cs: K.adapter_cols(X, V, S, Rp, want_colsum=True, out=out, cs=cs)))
    return cases


def kernels(reps, rounds):
    sets = {Rp: kernel_cases(Rp) for Rp in (32, 64)}
    times = {Rp: [[] for _ in sets[Rp]] for Rp in sets}
    for _ in range(rounds):
        for i in range(len(sets[32])):
            for Rp in (32, 64):
                times[Rp][i].append(timed(sets[Rp][i][3], reps))
    res = []
    for i in range(len(sets[32])):
        row = {"kernel": sets[32][i][0], **sets[32][i][1]}
        for Rp in (32, 64):
            name, _, nbytes, _ = sets[Rp][i]
            t = sorted(times[Rp][i])[len(times[Rp][i]) // 2]
            row["rp%d" % Rp] = {"us": round(t * 1e3, 2), "MB": round(nbytes / 1e6, 1), "GB_per_s": round(nbytes / t * 1e-6, 1)}
        res.append(row)
    del sets
    torch.cuda.empty_cache()
    return res


def steps(ranks, batch, n_steps, rounds):
    import bench
    from cara_b200 import kernels as K
    from cara_b200 import train as T
    dev = torch.device("cuda", 0)
    bench._install_init_module()
    x = torch.randn(batch, 3, 224, 224, device=dev)
    y = torch.randint(0, bench.NUM_CLASSES, (batch,), device=dev)
    graphs = {}
    for r in ranks:
        vit, opt = bench.build_model(dict(model="vit_base_patch16_224_in21k", rank=r), dev)
        graphs[r] = (T.GraphedStep(vit, opt, x, y), vit, opt)
        for _ in range(3):
            graphs[r][0](x, y)
    torch.cuda.synchronize()
    ms = {r: [] for r in ranks}
    sampler = bench.ClockSampler(0)
    sampler.start()
    for _ in range(rounds):
        for r in ranks:
            step = graphs[r][0]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n_steps):
                step(x, y)
            e1.record()
            torch.cuda.synchronize()
            ms[r].append(e0.elapsed_time(e1) / n_steps)
    clocks = sampler.stop()
    out = []
    for r in ranks:
        v = sorted(ms[r])
        med = v[len(v) // 2]
        out.append({"rank": r, "Rp": K.round_rank(r), "batch": batch, "step_ms_median": round(med, 3),
                    "step_ms_rounds": [round(t, 3) for t in ms[r]], "img_per_s": round(batch / med * 1e3, 1)})
    base = out[0]["step_ms_median"]
    for o in out:
        o["vs_rank16"] = round(o["step_ms_median"] / base, 4)
    del graphs
    torch.cuda.empty_cache()
    return out, clocks


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_rank64.json"))
    p.add_argument("--reps", type=int, default=20, help="timed passes per kernel and round")
    p.add_argument("--rounds", type=int, default=3, help="alternation rounds (kernels and steps)")
    p.add_argument("--steps", type=int, default=20, help="graph replays per rank and round")
    p.add_argument("--batch", type=int, default=256)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_time.py measures on the GPU; no CUDA device found")
    res = {"card": card(), "M": M, "l2": "overwritten (256 MB memset) before every timed kernel pass", "bytes": BYTES,
           "reps": a.reps, "rounds": a.rounds}
    res["kernels"] = kernels(a.reps, a.rounds)
    res["step"], res["step_clocks"] = steps((16, 32, 64), a.batch, a.steps, a.rounds)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that two builds can be compared by."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def test_dump_writes_loss_and_parameters(tmp_path):
    from cara_b200 import train as T
    g = torch.Generator().manual_seed(5)
    params = [("CP_A1", torch.nn.Parameter(torch.randn(6, 4, generator=g))),
              ("head.weight", torch.nn.Parameter(torch.randn(3, 5, generator=g)))]
    flat = T.FlatTrainable(params)
    flat.grad.copy_(torch.randn(flat.grad.shape, generator=g))
    opt = T.FusedAdamW(flat)
    bench.dump_outputs(str(tmp_path / "out"), bench.step_outputs(torch.tensor(2.5), opt))
    names = sorted(os.listdir(str(tmp_path / "out")))
    assert names == ["loss.npy", "param.CP_A1.npy", "param.head.weight.npy"]
    for n, p in params:
        got = np.load(str(tmp_path / "out" / ("param.%s.npy" % n)))
        assert got.dtype == np.float32 and np.array_equal(got, p.detach().numpy())
    assert np.load(str(tmp_path / "out" / "loss.npy")).tolist() == [2.5]


def _bench(steps, out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--batch", "4", "--no-cpu-baseline", "--dump-outputs", out_dir]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


@pytest.mark.gpu
def test_dumped_outputs_repeat_across_runs_and_follow_steps(tmp_path):
    """Same arguments, same seeded model and batches: two runs agree up to the order of the fp32 atomics of the factor
    gradients (the bars of test_graphed_step_matches_eager_steps).  One timed step fewer is one AdamW update fewer:
    about lr = 1e-3 per element of a head initialised at ~2e-2."""
    a = _bench(2, str(tmp_path / "a"))
    b = _bench(2, str(tmp_path / "b"))
    c = _bench(1, str(tmp_path / "c"))
    assert set(a) == set(b) == set(c) and "loss" in a and "param.CP_A1" in a and "param.head.weight" in a
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert abs(float(a["loss"][0]) - float(b["loss"][0])) < 2e-3
    for k in a:
        assert _rel(a[k], b[k]) < 1e-3, (k, _rel(a[k], b[k]))
    assert _rel(c["param.head.weight"], a["param.head.weight"]) > 1e-2

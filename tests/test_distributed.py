"""Multi-rank correctness of the data-parallel step (SURVEY 8e): N ranks on 1/N of the batch each, one sum
all-reduce of the flat CP+head gradient, the 1/N folded into AdamW's grad scale == one rank on the whole batch.

* CPU (gloo, world 2): the host logic -- shard_batch, FlatTrainable's gradient views, allreduce_grads, grad scale.
* GPU (NCCL, torchrun, one rank per GPU; skipped with fewer than 2 GPUs): the real CUDA step through GraphedStep, with
  the all-reduce and the AdamW kernel captured inside the CUDA graph and, again, launched eagerly.
"""
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import cara_oracle as O
from tests import _dist_workers as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_gloo_world2_flat_gradient_allreduce_equals_full_batch(tmp_path):
    import torch.multiprocessing as mp
    from cara_b200 import train as T
    world = 2
    mp.spawn(W.cpu_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    res = [torch.load(os.path.join(str(tmp_path), "rank%d.pt" % r)) for r in range(world)]
    assert [r["range"] for r in res] == [(0, 4), (4, 8)]
    # single process, full batch
    params = [(n, torch.nn.Parameter(t.clone())) for n, t in W._toy_params()]
    flat = T.FlatTrainable(params)
    g = torch.Generator().manual_seed(99)
    X, Y = torch.randn(8, 6, generator=g), torch.randint(0, 3, (8,), generator=g)
    flat.zero_grad()
    W._toy_loss(params, X, Y).backward()
    # the all-reduced buffer is the SUM of the shard gradients on every rank, and sum / world == the full-batch mean
    assert torch.equal(res[0]["summed_grad"], res[1]["summed_grad"])
    assert torch.allclose(res[0]["summed_grad"], res[0]["local_grad"] + res[1]["local_grad"], rtol=0, atol=1e-7)
    assert torch.allclose(res[0]["summed_grad"] / world, flat.grad, rtol=1e-5, atol=1e-7)
    assert not torch.allclose(res[0]["local_grad"], res[1]["local_grad"])     # the shards really differ
    for n, p in params:
        a, b = flat.slices[n]
        want = O.adamw_update(p.detach(), flat.grad[a:b].view(p.shape), torch.zeros_like(p), torch.zeros_like(p), 1)[0]
        for r in res:
            assert torch.allclose(r["params"][n], want, rtol=1e-5, atol=1e-7), n
    with pytest.raises(ValueError):
        T.shard_batch(9, 0, 2)


def _torchrun(nproc, extra_env, log_path, limit=420):
    """torchrun of tests/_dist_workers.py; output goes to a FILE (no pipes that a lingering grandchild could keep open)
    and the whole process group is killed when the time limit passes."""
    import signal
    env = dict(os.environ)
    env.update(extra_env)
    cmd = [sys.executable, "-u", "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "_dist_workers.py")]
    with open(log_path, "w") as log:
        proc = subprocess.Popen(cmd, env=env, cwd=ROOT, stdout=log, stderr=subprocess.STDOUT, start_new_session=True)
        try:
            rc = proc.wait(timeout=limit)
        except subprocess.TimeoutExpired:
            os.killpg(proc.pid, signal.SIGKILL)
            proc.wait()
            rc = -9
    return rc, open(log_path).read()


@pytest.mark.gpu
@pytest.mark.parametrize("captured", ["0", "1"])
def test_two_gpu_half_batches_equal_one_gpu_full_batch(captured, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rc, out = _torchrun(2, {"CARA_GRAPH_COLLECTIVE": captured}, os.path.join(str(tmp_path), "dist.log"))
    print(out[-3000:])
    assert rc == 0 and "DIST_OK" in out, out[-3000:]

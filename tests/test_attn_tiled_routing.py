"""Which attention kernels ops.AttnCoreFunction runs (no GPU): D = 80 stays on the whole-head kernels up to their
shared-memory limits (forward N <= 432, backward N <= 320) and takes the key-tiled kernels above them; D = 64 never
takes the tiled ones."""
import pytest
import torch

from cara_b200 import kernels as K
from cara_b200 import ops


class _Recorder:
    """Stands in for the four attention wrappers: records which were called."""

    def __init__(self, monkeypatch):
        self.calls = []
        monkeypatch.setattr(K, "attn_fwd", self._fwd("attn_fwd"))
        monkeypatch.setattr(K, "attn_tiled_fwd", self._fwd("attn_tiled_fwd"))
        monkeypatch.setattr(K, "attn_bwd", self._bwd("attn_bwd"))
        monkeypatch.setattr(K, "attn_tiled_bwd", self._bwd("attn_tiled_bwd"))

    def _fwd(self, name):
        def fwd(qkv, B, N, H, D, scale, train=True):
            self.calls.append(name)
            o = torch.zeros(B * N, H * D)
            return o, (torch.zeros_like(o) if train else None), (torch.zeros(B, H, N) if train else None)
        return fwd

    def _bwd(self, name):
        def bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, scale, delta=None):
            self.calls.append(name)
            assert o is not None and o_lo is not None and lse is not None
            return torch.zeros_like(qkv)
        return bwd


def _run(N, D, B=2, H=2, train=True):
    qkv = torch.zeros(B * N * 3 * H * D, requires_grad=train)
    o = ops.AttnCoreFunction.apply(qkv, B, N, H, D, D ** -0.5)
    if train:
        o.sum().backward()


def test_whole_head_limits_live_in_one_place():
    assert K.D80_WHOLE_HEAD_MAX_N == {"fwd": 432, "bwd": 320}


@pytest.mark.parametrize("N,D,expected", [
    (257, 80, ["attn_fwd", "attn_bwd"]),                 # ViT-H/14 @224: the launches it always had
    (320, 80, ["attn_fwd", "attn_bwd"]),                 # the whole-head backward's limit
    (321, 80, ["attn_fwd", "attn_tiled_bwd"]),           # whole-head forward feeds the tiled backward
    (432, 80, ["attn_fwd", "attn_tiled_bwd"]),           # the whole-head forward's limit
    (433, 80, ["attn_tiled_fwd", "attn_tiled_bwd"]),
    (577, 80, ["attn_tiled_fwd", "attn_tiled_bwd"]),     # ViT-H/14 @336
    (577, 64, ["attn_fwd", "attn_bwd"]),                 # D = 64: the tcgen05 kernels behind attn_fwd / attn_bwd
])
def test_attention_core_routing(monkeypatch, N, D, expected):
    rec = _Recorder(monkeypatch)
    _run(N, D)
    assert rec.calls == expected


@pytest.mark.parametrize("N,expected", [(432, "attn_fwd"), (433, "attn_tiled_fwd")])
def test_inference_routing(monkeypatch, N, expected):
    rec = _Recorder(monkeypatch)
    with torch.no_grad():
        _run(N, 80, train=False)
    assert rec.calls == [expected]

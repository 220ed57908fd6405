"""Host-side handling of the adapter rank (no GPU): the padded rank the bf16 kernels run at, the refusal above 64, and
which kernels an Rp = 64 projection is routed to when CARA_SIDE_TILES=1 asks for the GEMM's side tiles."""
import pytest
import torch

from cara_b200 import kernels as K
from cara_b200 import ops


def test_round_rank_pads_to_16_32_or_64():
    assert [K.round_rank(r) for r in (1, 8, 12, 16)] == [16] * 4
    assert [K.round_rank(r) for r in (17, 24, 32)] == [32] * 3
    assert [K.round_rank(r) for r in (33, 40, 48, 63, 64)] == [64] * 5
    assert K.MAX_RANK == 64


@pytest.mark.parametrize("r", [65, 96, 128])
def test_round_rank_refuses_above_64(r):
    with pytest.raises(ValueError, match="64"):
        K.round_rank(r)


def test_staging_refuses_rank65_with_a_message_naming_64():
    from cara_b200 import staging
    from cara_b200.vit import create_model
    from src.cara.cara import cara
    vit = create_model("vit_base_patch16_224_in21k", depth=1)
    vit = cara({"model": vit, "rank": 65, "scale": 1.0, "l_mu": 1.0, "l_std": 0.0})
    with pytest.raises(NotImplementedError, match="rank > 64"):
        staging.staged(vit)


class _Recorder:
    """Stands in for the kernel wrappers: records which were called and with which side tiles."""

    def __init__(self, monkeypatch, rp, slices=1):
        self.calls = []
        self.rp, self.slices = rp, slices
        monkeypatch.setattr(K, "side_tiles", True)
        monkeypatch.setattr(K, "adapter_rows_fwd", self.rows_fwd)
        monkeypatch.setattr(K, "adapter_rows_bwd", self.rows_bwd)
        monkeypatch.setattr(K, "adapter_cols", self.cols)
        monkeypatch.setattr(K, "gemm_cp", self.gemm)

    def rows_fwd(self, x, a_t2, scales):
        self.calls.append("rows_fwd")
        return torch.zeros(x.shape[0], self.rp), torch.zeros(x.shape[0], self.slices * 3 * self.rp)

    def rows_bwd(self, G, b_t2, scales, T, dsc=None):
        self.calls.append("rows_bwd")
        return torch.zeros(G.shape[0], 3 * self.rp), dsc

    def cols(self, *a, **kw):
        self.calls.append("cols")

    def gemm(self, a0, b0, side=None, **kw):
        self.calls.append("gemm+side" if side is not None else "gemm")
        return torch.zeros(a0.shape[0], b0.shape[0])


def _operands(rp, R, slices=1, K_in=64, N=64):
    z = lambda *s: torch.zeros(*s)                                            # noqa: E731
    return ops.AdapterOperands(z(K_in, 3 * rp), z(2 * rp, K_in), z(N // slices, 3 * rp), z(2 * rp, N // slices),
                               z(slices, rp), R)


class _Frozen:
    def __init__(self, K_in=64, N=64):
        self.w, self.wt, self.bias = torch.zeros(N, K_in), torch.zeros(K_in, N), None


@pytest.mark.parametrize("rp,R,side", [(16, 8, True), (32, 32, True), (64, 33, False), (64, 64, False)])
def test_side_tile_switch_routes_rp64_to_the_rows_pass(monkeypatch, rp, R, side):
    """CARA_SIDE_TILES=1: Rp = 16 / 32 projections get the rank-R row contraction as side tiles of their GEMM; Rp = 64
    ones (not covered by the side tiles) keep the stand-alone rows pass, forward and backward."""
    rec = _Recorder(monkeypatch, rp)
    x = torch.zeros(10, 64)
    ops._cp_linear_fwd(x, _Frozen(), None, _operands(rp, R))
    assert rec.calls == (["gemm+side"] if side else ["rows_fwd", "gemm"])
    rec.calls.clear()
    T, U = torch.zeros(10, rp), torch.zeros(10, 3 * rp)
    ops._cp_linear_bwd(torch.zeros(10, 64), x, _Frozen(), _operands(rp, R), T, U, True, False)
    assert rec.calls == (["cols", "gemm+side", "cols"] if side else ["rows_bwd", "cols", "gemm", "cols"])


def test_without_the_switch_every_rank_takes_the_rows_pass(monkeypatch):
    rec = _Recorder(monkeypatch, 64)
    monkeypatch.setattr(K, "side_tiles", False)
    ops._cp_linear_fwd(torch.zeros(10, 64), _Frozen(), None, _operands(64, 64))
    assert rec.calls == ["rows_fwd", "gemm"]

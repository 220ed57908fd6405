"""The attention kernels that run at 224 px, per head against an fp64 reference, at every tile boundary they have:
* D = 64, N <= 256: attn_fwd_tc8_kernel + attn_bwd_tc_kernel (csrc/attention_tc.cu, tcgen05; ViT-B/L/16).
  Boundaries: 16-row padding, the second 128-row query box (read from row 128 whatever npad is), the two softmax
  column halves of the forward, the backward's prefetch of the next head's Q/K (only while a second Q/K pair fits in
  shared memory: N <= 208) and both persistent grids (forward min(B H, 296) CTAs, backward min(B H, 148)).
* D = 80: attn_fwd_kernel<80> / attn_bwd_kernel<80> (csrc/attention.cu, mma.sync, the whole head in shared memory;
  ViT-H/14).  Boundaries: the 64-key (forward, dQ) and 64-query (dK/dV) chunks with a remainder of 1, 2 or 3 16-row
  steps, and the shared-memory limits N <= 432 (forward) and N <= 320 (backward)."""
import math

import pytest
import torch

from tests._attn_ref import check

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def K():
    from cara_b200 import kernels
    return kernels


def _qkv(B, N, H, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)


def _npad(N):
    return (N + 15) // 16 * 16


# ------------------------------------------------------------------------------------------- D = 64, tcgen05, N <= 256
@pytest.mark.parametrize("N", [1, 2, 15, 16, 17,                # one 16-row step: npad = 16, 16, 16, 16, 32
                               127, 128, 129,                   # one 128-row query / key tile, and one row of a second
                               143, 144, 145,                   # second tile of 16 / 16 / 17 rows
                               197,                             # ViT-B/16 @224
                               208, 209,                        # largest N with the Q/K prefetch, smallest without
                               240, 255, 256])
def test_tc_attention_matches_fp64(K, N):
    B, H = 3, 4
    check(K, _qkv(B, N, H, 64, N), B, N, H)


@pytest.mark.parametrize("B,N,H", [(37, 197, 4),                # 148 heads: one per backward CTA
                                   (149, 129, 1),               # 149: one backward CTA takes a second head
                                   (37, 208, 8),                # 296: one per forward CTA (prefetching backward)
                                   (99, 209, 3)])               # 297: one forward CTA takes a second head
def test_tc_attention_persistent_grid_edges(K, B, N, H):
    check(K, _qkv(B, N, H, 64, B * H), B, N, H)


def test_tc_attention_benchmark_shape_every_sample(K):
    """The benchmark's shape (ViT-B/16 @224, batch 256): 3,072 heads, 10 or 11 per forward CTA and 20 or 21 per
    backward CTA."""
    B, N, H = 256, 197, 12
    check(K, _qkv(B, N, H, 64, 7), B, N, H)
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------- D = 80, mma.sync
# (npad / 16) % 4 = the 16-row steps left after the last full 64-key chunk of the forward / dQ pass and the last
# 64-query chunk of the dK/dV pass
@pytest.mark.parametrize("N", [1, 16, 17, 48,                   # remainder 1, 1, 2, 3 with no full chunk
                               63, 64, 65, 96, 112,             # 0, 0, 1, 2, 3 after one chunk
                               127, 128, 129,                   # 0, 0, 1
                               197, 257,                        # ViT-H/14 @224: 1 (npad 208), 1 (npad 272)
                               320])                            # the backward's shared-memory limit, remainder 0
def test_d80_attention_matches_fp64(K, N):
    B, H = 3, 2
    check(K, _qkv(B, N, H, 80, N), B, N, H)


@pytest.mark.parametrize("N", [401,                             # remainder 2 (npad 416), above the backward's limit
                               432])                            # the forward's shared-memory limit, remainder 3
def test_d80_forward_only_matches_fp64(K, N):
    B, H = 2, 2
    check(K, _qkv(B, N, H, 80, N), B, N, H, backward=False)


def test_d80_shared_memory_limits(K):
    """Beyond the limits the calls fail with an error before anything is launched."""
    from cara_b200 import _lib as L
    B, H, D = 2, 2, 80
    qkv = _qkv(B, 433, H, D, 1)
    with pytest.raises(L.CaraLibraryError):
        K.attn_fwd(qkv.view(-1), B, 433, H, D, D ** -0.5)
    N = 321                                                     # forward fits, backward does not
    qkv = _qkv(B, N, H, D, 2)
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, D ** -0.5)
    d_o = torch.randn(B * N, H * D, device="cuda").to(BF16)
    with pytest.raises(L.CaraLibraryError):
        K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, D ** -0.5)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------- both paths
@pytest.mark.parametrize("D,N", [(64, 17), (64, 129), (64, 197), (64, 255), (80, 65), (80, 197)])
def test_no_leakage_across_samples(K, D, N):
    """Sample 1's K and V scaled by 50: a key or query row of sample 1 that a box of sample 0 reads past its N, and
    that is not masked, would dominate sample 0's softmax.  Samples 0 and 2 still match their own references."""
    B, H = 3, 4
    g = torch.Generator(device="cuda").manual_seed(9)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g)
    qkv[1, :, 1:] *= 50.0
    check(K, qkv.to(BF16).contiguous(), B, N, H, samples=[0, 2])


def _peaked(B, N, H, D, late, early, amp, seed):
    """Even query rows = amp u, odd rows = amp w (u . w = 0, |u|^2 = |w|^2 = D); keys ``late`` = amp u + spread and keys
    ``early`` = amp w + spread, every other entry 0.3 N(0, 1).  Even rows then peak on ``late`` and odd rows on
    ``early``; the spread keeps a row's probability from sitting on one key (a one-hot row has dq = 0 exactly).
    Built on the CPU, so that the checks below run on exactly the data the kernels get.  Returns (qkv on the GPU,
    base-2 scaled scores [B,H,N,N] fp64)."""
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, N, 3, H, D, generator=g) * 0.3
    u = torch.ones(D); u[D // 2:] = -1.0
    w = torch.ones(D); w[1::2] = -1.0
    spread = lambda n: 0.5 * torch.randn(B, n, H, D, generator=g)           # noqa: E731
    qkv[:, 0::2, 0] = amp * u
    qkv[:, late, 1] = amp * u + spread(late.stop - late.start)
    qkv[:, 1::2, 0] = amp * w
    qkv[:, early, 1] = amp * w + spread(early.stop - early.start)
    qkv = qkv.to(BF16)
    s = torch.einsum("bnhd,bmhd->bhnm", qkv[:, :, 0].double(), qkv[:, :, 1].double()) * D ** -0.5 / math.log(2.0)
    return qkv.cuda().contiguous(), s


def _assert_peaks(s, late, early, min_gap):
    top = s.argmax(-1)
    assert bool(((top[:, :, 0::2] >= late.start) & (top[:, :, 0::2] < late.stop)).all())
    assert bool(((top[:, :, 1::2] >= early.start) & (top[:, :, 1::2] < early.stop)).all())
    outside = torch.ones(s.shape[-1], dtype=torch.bool)
    outside[late] = False
    gap_late = s[:, :, 0::2, late].amax(-1) - s[:, :, 0::2][..., outside].amax(-1)
    outside = torch.ones(s.shape[-1], dtype=torch.bool)
    outside[early] = False
    gap_early = s[:, :, 1::2, early].amax(-1) - s[:, :, 1::2][..., outside].amax(-1)
    assert float(gap_late.min()) >= min_gap and float(gap_early.min()) >= min_gap, (gap_late.min(), gap_early.min())
    p = torch.softmax(s * math.log(2.0), -1)
    assert float(p.amax(-1).max()) < 0.99                               # no row is one-hot


@pytest.mark.parametrize("N", [197, 255])
def test_tc_softmax_peak_in_either_column_half(K, N):
    """D = 64 forward: each of two warps per query row takes the maximum over its half of the key columns, [0, split)
    or [split, npad).  Rows whose maximum is in the second half lie >= 30 (base 2) above everything in the first, and
    the other way round: a row maximum that does not combine both halves overflows or loses the row."""
    B, H, D = 2, 12, 64
    npad = _npad(N)
    split = ((npad // 16 + 1) // 2) * 16
    late, early = slice(split, N), slice(0, split)
    qkv, s = _peaked(B, N, H, D, late, early, 2.0, 5)
    _assert_peaks(s, late, early, 30.0)
    check(K, qkv, B, N, H)


@pytest.mark.parametrize("N,amp,min_gap", [(197, 2.0, 30.0),         # keys 192..196 of the last chunk
                                           (257, 0.9, 8.0)])         # key 256 alone: a smaller lead keeps it from
                                                                     # holding the whole row
def test_d80_online_softmax_peak_in_last_chunk(K, N, amp, min_gap):
    """D = 80 forward: rows whose maximum sits in the remainder chunk after the last full 64-key chunk -- the running
    maximum and the rescaling of O / l must absorb it there -- and rows whose maximum sits in the first chunk."""
    B, H, D = 2, 4, 80
    k_last = _npad(N) // 64 * 64
    late, early = slice(k_last, N), slice(0, 64)
    qkv, s = _peaked(B, N, H, D, late, early, amp, 6)
    _assert_peaks(s, late, early, min_gap)
    check(K, qkv, B, N, H)


@pytest.mark.parametrize("B,N,H,D", [(256, 197, 12, 64),           # the benchmark's 3,072 heads
                                     (8, 257, 16, 80)])             # ViT-H/14 @224
def test_attention_is_deterministic(K, B, N, H, D):
    scale = D ** -0.5
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
    runs = []
    for _ in range(2):
        o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale)
        runs.append((o, o_lo, lse, K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, scale)))
    for name, a, b in zip(("o", "o_lo", "lse", "dqkv"), *runs):
        assert torch.equal(a, b), name

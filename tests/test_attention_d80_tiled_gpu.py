"""The key-tiled D = 80 attention kernels (csrc/attention_tiled.cu: ViT-H/14 at any sequence length) per head against
an fp64 reference at every window boundary, bit for bit against the whole-head kernels (csrc/attention.cu) wherever
those run, and the model above 224 px against the CPU oracle and through the entry point.

Boundaries: the 64-key (forward, dQ) and 64-query (dK/dV) windows with a remainder of 0-3 16-row steps, the forward's
128-query tiles (N = 127 / 128 / 129, 257), the backward's 64-row tiles, one window (N <= 64) and many (N = 1370)."""
import os
import types

import pytest
import torch

from oracle import cara_oracle as O
from tests._attn_ref import check
from tests.test_attention_core_gpu import _assert_peaks, _peaked

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
D = 80
VIT_H14 = dict(embed_dim=1280, num_heads=16, patch=14)


@pytest.fixture(scope="module")
def K():
    from cara_b200 import kernels
    return kernels


@pytest.fixture(scope="module")
def tiled(K):
    """kernels with attn_fwd / attn_bwd bound to the tiled entry points, for tests._attn_ref.check"""
    return types.SimpleNamespace(attn_fwd=K.attn_tiled_fwd, attn_bwd=K.attn_tiled_bwd)


def _qkv(B, N, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)


# (npad / 16) % 4 = the 16-row steps after the last full window
SMALL_N = [1, 15, 16, 17,               # one window, remainder 1, 1, 1, 2
           48, 63, 64, 65,              # 3, 0, 0, 1
           127, 128, 129,               # 0, 0, 1; 129 opens the forward's second 128-query tile
           192, 193,                    # 0, 1
           257]                         # ViT-H/14 @224: 1


@pytest.mark.parametrize("N", SMALL_N + [321,            # ViT-H/14 @252 has 325 tokens; 321 is the first N the
                                                         # whole-head backward refuses
                                         433, 449])      # the first N the whole-head forward refuses, and one window on
def test_tiled_matches_fp64(tiled, N):
    B, H = 3, 2
    check(tiled, _qkv(B, N, H, N), B, N, H)


@pytest.mark.parametrize("B,N,H", [(2, 577, 4),         # ViT-H/14 @336
                                   (1, 1025, 2),        # @448
                                   (1, 1370, 1)])       # @518
def test_tiled_matches_fp64_long(tiled, B, N, H):
    check(tiled, _qkv(B, N, H, N), B, N, H)


@pytest.mark.parametrize("N", SMALL_N + [321, 401, 432])
def test_tiled_forward_is_bit_identical_to_whole_head(K, N):
    B, H = 3, 4
    qkv = _qkv(B, N, H, N + 1).view(-1)
    for train in (True, False):
        mine = K.attn_tiled_fwd(qkv, B, N, H, D, D ** -0.5, train=train)
        theirs = K.attn_fwd(qkv, B, N, H, D, D ** -0.5, train=train)
        for name, a, b in zip(("o", "o_lo", "lse"), mine, theirs):
            assert (a is None and b is None) or torch.equal(a, b), (N, train, name)


@pytest.mark.parametrize("N", SMALL_N + [320])
def test_tiled_backward_is_bit_identical_to_whole_head(K, N):
    B, H = 3, 4
    qkv = _qkv(B, N, H, N + 2).view(-1)
    o, o_lo, lse = K.attn_fwd(qkv, B, N, H, D, D ** -0.5)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(N)).to(BF16)
    mine = K.attn_tiled_bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, D ** -0.5)
    theirs = K.attn_bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, D ** -0.5)
    assert torch.equal(mine, theirs), N


@pytest.mark.parametrize("N", [321, 325, 401, 432])
def test_whole_head_forward_then_tiled_backward_matches_fp64(K, N):
    """What fine-tuning at 252-280 px runs: the forward still fits the whole-head kernel, the backward does not."""
    B, H = 3, 2
    mixed = types.SimpleNamespace(attn_fwd=K.attn_fwd, attn_bwd=K.attn_tiled_bwd)
    check(mixed, _qkv(B, N, H, N + 3), B, N, H)


@pytest.mark.parametrize("N", [449, 577])
def test_no_leakage_across_samples(tiled, N):
    """Sample 1's K and V scaled by 50: a window of sample 0 that read rows of sample 1 past its N, or an unmasked
    zero-filled row, would dominate sample 0's softmax.  Samples 0 and 2 still match their own references."""
    B, H = 3, 4
    g = torch.Generator(device="cuda").manual_seed(9)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g)
    qkv[1, :, 1:] *= 50.0
    check(tiled, qkv.to(BF16).contiguous(), B, N, H, samples=[0, 2])


def test_online_softmax_peak_in_last_and_first_window(tiled):
    """N = 577: even rows peak on key 576, alone in the last (partial) window, so the running maximum and the rescaling
    of O / l must absorb it in the last step; odd rows peak in the first window."""
    B, N, H = 2, 577, 4
    k_last = (N + 15) // 16 * 16 // 64 * 64
    late, early = slice(k_last, N), slice(0, 64)
    qkv, s = _peaked(B, N, H, D, late, early, 1.0, 6)
    _assert_peaks(s, late, early, 8.0)
    check(tiled, qkv, B, N, H)


def test_tiled_is_deterministic(K):
    B, N, H = 8, 577, 16
    scale = D ** -0.5
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
    runs = []
    for _ in range(2):
        o, o_lo, lse = K.attn_tiled_fwd(qkv.view(-1), B, N, H, D, scale)
        runs.append((o, o_lo, lse, K.attn_tiled_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, scale)))
    for name, a, b in zip(("o", "o_lo", "lse", "dqkv"), *runs):
        assert torch.equal(a, b), name


def test_tiled_entry_errors(K):
    """D != 80, N = 0 and a missing o_lo fail with an error before anything is launched."""
    from cara_b200 import _lib as L
    B, N, H = 2, 577, 2
    q64 = torch.randn(B, N, 3, H, 64, device="cuda").to(BF16).view(-1)
    with pytest.raises(L.CaraLibraryError, match="D = 80"):
        K.attn_tiled_fwd(q64, B, N, H, 64, 0.125)
    o64 = torch.zeros(B * N, H * 64, device="cuda", dtype=BF16)
    lse64 = torch.zeros(B, H, N, device="cuda")
    with pytest.raises(L.CaraLibraryError, match="D = 80"):
        K.attn_tiled_bwd(q64, o64, o64, lse64, o64, B, N, H, 64, 0.125)
    with pytest.raises(L.CaraLibraryError, match="N, H >= 1"):
        K.attn_tiled_fwd(torch.zeros(0, device="cuda", dtype=BF16), B, 0, H, D, D ** -0.5)
    qkv = _qkv(B, N, H, 1).view(-1)
    o, o_lo, lse = K.attn_tiled_fwd(qkv, B, N, H, D, D ** -0.5)
    d_o = torch.randn(B * N, H * D, device="cuda").to(BF16)
    with pytest.raises(L.CaraLibraryError, match="o_lo"):
        K.attn_tiled_bwd(qkv, o, None, lse, d_o, B, N, H, D, D ** -0.5)
    torch.cuda.synchronize()


@pytest.mark.parametrize("img,tokens,tiled_fwd", [(280, 401, False),    # whole-head forward, tiled backward
                                                  (336, 577, True)])
def test_reduced_depth_vit_h14_above_224px_vs_oracle(monkeypatch, K, img, tokens, tiled_fwd):
    from tests.test_parity_gpu import build, check_against, run_step
    calls = []
    for name in ("attn_tiled_fwd", "attn_tiled_bwd"):
        fn = getattr(K, name)
        monkeypatch.setattr(K, name, lambda *a, _fn=fn, _name=name, **kw: calls.append(_name) or _fn(*a, **kw))
    g = O.Geometry(img=img, depth=2, rank=32, num_classes=100, **VIT_H14)
    assert g.tokens == tokens
    vit, st = build(g, 1.0)
    vit.eval()
    x, y = O.synthetic_batch(g, 2)
    logits, loss, grads = run_step(vit, x, y)
    assert calls.count("attn_tiled_fwd") == (2 if tiled_fwd else 0) and calls.count("attn_tiled_bwd") == 2, calls
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, 1.0)
    # two blocks: the reduced-depth bars of tests/test_parity_gpu.py (logits 1.5e-2, gradient cosine 0.999)
    e, worst = check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "ViT-H/14 @%d" % img,
                             logits_tol=1.5e-2)
    print("ViT-H/14 depth 2 r32 @%d px: logits rel %.3e, worst grad cosine %.6f (%s)" % (img, e, worst[0], worst[1]))


def test_vit_cp_cli_vit_h14_336px_trains_saves_and_evaluates(tmp_path):
    import glob
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root)
    base = [sys.executable, os.path.join(root, "image_classification", "vit_cp.py"), "--model=vit_huge_patch14_224_in21k",
            "--img-size=336", "--dataset=cifar", "--dim=8", "--synthetic"]
    r = subprocess.run(base + ["--epochs=1", "--batch-size=16"], cwd=str(tmp_path), env=env, capture_output=True,
                       text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "e: 0, l:" in r.stdout and "Accuracy:" in r.stdout, r.stdout[-2000:]
    loss = float(r.stdout.split("e: 0, l:")[1].split(",")[0])
    assert 3.0 < loss < 7.0, loss
    ckpts = glob.glob(os.path.join(str(tmp_path), "vit_cifar_*_seed_*.pt"))
    assert len(ckpts) == 1, (ckpts, r.stdout[-2000:])
    assert torch.load(ckpts[0], map_location="cpu", mmap=True)["pos_embed"].shape[1] == 577
    acc_train_run = float(r.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    e = subprocess.run(base + ["--evaluate=" + ckpts[0]], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                       timeout=1800)
    assert e.returncode == 0 and "Only evaluation" in e.stdout, e.stderr[-3000:]
    acc_eval = float(e.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    assert abs(acc_eval - acc_train_run) <= 2.0 / 512 + 1e-9, (acc_eval, acc_train_run)

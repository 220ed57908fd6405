"""The key-tiled tcgen05 attention kernels (csrc/attention_long.cu: D = 64, N > 256) against an fp64 reference, per
head, at the tail cases N % 128 in {1, 127, 0} and the token counts of ViT-B/L/16 above 224 px; and the model at
384 px against the CPU oracle, through the entry point and the GPU preprocessor."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import cara_oracle as O
from tests._attn_ref import check

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
D = 64


@pytest.fixture(scope="module")
def K():
    from cara_b200 import kernels
    return kernels


@pytest.mark.parametrize("B,N,H", [(2, 257, 12),     # N % 128 = 1: the last key / query tile holds one row
                                   (3, 383, 4),      # N % 128 = 127
                                   (2, 385, 12), (2, 401, 12),
                                   (4, 512, 4),      # N % 128 = 0
                                   (8, 577, 12),     # ViT-B/16 @384
                                   (2, 577, 16),     # ViT-L/16 @384
                                   (2, 785, 12),     # ViT-B/16 @448
                                   (1, 1025, 12),
                                   (64, 577, 12)])   # 3,840 work items: every persistent CTA walks over many
def test_long_attention_matches_fp64(K, B, N, H):
    g = torch.Generator(device="cuda").manual_seed(N + B)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    check(K, qkv, B, N, H)


@pytest.mark.parametrize("N", [512, 700])
def test_online_softmax_peak_in_last_or_first_tile(K, N):
    """Rows whose maximum score sits in the LAST key tile, >= 30 (base 2) above every earlier tile -- the running max
    and the rescaling of the partial O / l must absorb it -- and rows whose maximum sits in the first tile.  The keys of
    the peak tile spread over a few units, so that no row is one-hot (a one-hot row has dq = 0 exactly)."""
    B, H = 2, 12
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g) * 0.3
    u = torch.ones(D, device="cuda"); u[D // 2:] = -1.0                    # u . w = 0
    w = torch.ones(D, device="cuda"); w[1::2] = -1.0
    last = (N - 1) // 128 * 128                                             # first key of the last tile
    spread = lambda n: 0.5 * torch.randn(B, n, H, D, device="cuda", generator=g)   # noqa: E731
    # peak scores ~ 2 * 2 * 64 / 8 = 32 (natural) = 46 (base 2) +- a few; every other pair stays around 0 +- 1.5
    qkv[:, 0::2, 0] = 2.0 * u
    qkv[:, last:, 1] = 2.0 * u + spread(N - last)
    qkv[:, 1::2, 0] = 2.0 * w
    qkv[:, :128, 1] = 2.0 * w + spread(128)
    qkv = qkv.to(BF16).contiguous()
    s = torch.einsum("bnhd,bmhd->bhnm", qkv[:, :, 0].float(), qkv[:, :, 1].float()) * D ** -0.5 / math.log(2.0)
    top = s.argmax(-1)
    assert bool((top[:, :, 0::2] >= last).all()) and bool((top[:, :, 1::2] < 128).all())
    gap_last = s[:, :, 0::2, last:].amax(-1) - s[:, :, 0::2, :last].amax(-1)
    gap_first = s[:, :, 1::2, :128].amax(-1) - s[:, :, 1::2, 128:].amax(-1)
    assert float(gap_last.min()) >= 30.0 and float(gap_first.min()) >= 30.0
    check(K, qkv, B, N, H)


def test_no_leakage_across_samples(K):
    """Sample 1's K and V scaled by 50: a 128-row box of sample 0 that runs into sample 1, or an unmasked row of it,
    would dominate sample 0's softmax.  Samples 0 and 2 still match their own references."""
    B, N, H = 3, 577, 12
    g = torch.Generator(device="cuda").manual_seed(9)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g)
    qkv[1, :, 1:] *= 50.0
    check(K, qkv.to(BF16).contiguous(), B, N, H, samples=[0, 2])


def test_long_attention_is_deterministic(K):
    B, N, H = 8, 577, 12
    scale = D ** -0.5
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
    runs = []
    for _ in range(2):
        o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale)
        runs.append((o, o_lo, lse, K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, scale)))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_gemm_delta_epilogue_feeds_long_attention_backward(K):
    """EPI_DELTA at N = 577: the output projection's dX GEMM writes delta, the long backward consumes it (o == NULL)
    and equals the backward that runs its own pre-pass."""
    from cara_b200 import _lib as L
    B, N, H, R = 3, 577, 12, 16
    g = torch.Generator(device="cuda").manual_seed(11)
    C, M = H * D, B * N
    G = (torch.randn(M, C, device="cuda", generator=g) * 0.5).to(BF16)
    Wt = (torch.randn(C, C, device="cuda", generator=g) * 0.03).to(BF16)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, D ** -0.5)
    a1 = (torch.randn(M, 3 * R, device="cuda", generator=g) * 0.3).to(BF16)
    b1 = (torch.randn(C, 3 * R, device="cuda", generator=g) * 0.1).to(BF16)
    assert K.attn_delta_fusable(N, D)
    delta = torch.full((B, H, N), float("nan"), device="cuda")
    d_o = K.gemm_cp(G, Wt, a1=a1, b1=b1, epi=L.EPI_DELTA, delta=(o, o_lo, delta, N))
    ref = (d_o.float() * (o.float() + o_lo.float())).view(B, N, H, D).sum(-1).permute(0, 2, 1)
    assert torch.isfinite(delta).all()
    assert float((delta - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    mine = K.attn_bwd(qkv.view(-1), None, None, lse, d_o, B, N, H, D, D ** -0.5, delta=delta)
    theirs = K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, D ** -0.5)
    a, b = mine.float().double(), theirs.float().double()
    assert float((a - b).norm() / b.norm()) < 1e-3


@pytest.mark.parametrize("geom", [dict(depth=2, rank=8, num_classes=10),
                                  dict(embed_dim=1024, depth=2, num_heads=16, rank=32, num_classes=100)])
def test_reduced_depth_384px_vs_oracle(geom):
    from tests.test_parity_gpu import build, check_against, run_step
    g = O.Geometry(img=384, **geom)
    assert g.tokens == 577
    vit, st = build(g, 1.0)
    vit.eval()
    x, y = O.synthetic_batch(g, 2)
    logits, loss, grads = run_step(vit, x, y)
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, 1.0)
    check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "384 px " + str(geom), logits_tol=1.5e-2)


def test_vitb_r16_384px_full_depth_vs_oracle():
    from tests.test_parity_gpu import build, check_against, run_step
    g = O.Geometry(img=384, depth=12, rank=16, num_classes=100)
    vit, st = build(g, 1.0)
    vit.eval()
    x, y = O.synthetic_batch(g, 2)
    logits, loss, grads = run_step(vit, x, y)
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, 1.0)
    e, worst = check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "ViT-B/16 r16 @384")
    print("ViT-B/16 r16 @384 px: logits rel %.3e, worst grad cosine %.6f (%s)" % (e, worst[0], worst[1]))


def test_vit_cp_cli_384px_trains_saves_and_evaluates(tmp_path):
    import glob
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root)
    base = [sys.executable, os.path.join(root, "image_classification", "vit_cp.py"), "--dataset=cifar", "--dim=8",
            "--synthetic", "--img-size=384"]
    r = subprocess.run(base + ["--epochs=1", "--batch-size=16"], cwd=str(tmp_path), env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "e: 0, l:" in r.stdout and "Accuracy:" in r.stdout, r.stdout[-2000:]
    loss = float(r.stdout.split("e: 0, l:")[1].split(",")[0])
    assert 3.0 < loss < 7.0, loss
    ckpts = glob.glob(os.path.join(str(tmp_path), "vit_cifar_*_seed_*.pt"))
    assert len(ckpts) == 1, (ckpts, r.stdout[-2000:])
    assert torch.load(ckpts[0], map_location="cpu")["pos_embed"].shape[1] == 577
    acc_train_run = float(r.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    e = subprocess.run(base + ["--evaluate=" + ckpts[0]], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                       timeout=900)
    assert e.returncode == 0 and "Only evaluation" in e.stdout, e.stderr[-3000:]
    acc_eval = float(e.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    assert abs(acc_eval - acc_train_run) <= 2.0 / 512 + 1e-9, (acc_eval, acc_train_run)


def test_gpu_preprocess_384_is_bit_identical():
    from cara_b200.preprocess import GpuPreprocessor, resize_reference
    rng = np.random.default_rng(4)
    pre = GpuPreprocessor("cuda:0", size=384)
    for h, w in [(500, 375), (32, 32), (384, 384), (640, 480)]:
        imgs = rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
        out, u8 = pre(imgs, return_uint8=True)
        assert out.shape == (2, 3, 384, 384) and u8.shape == (2, 384, 384, 3)
        for i in range(2):
            assert np.array_equal(u8[i].cpu().numpy(), resize_reference(imgs[i], 384, 384)), (h, w, i)

"""CaRA adapters of rank 33..64 (padded rank Rp = 64) on the fused bf16 path, on the GPU.

Kernel level: the Rp = 64 skinny kernels (rows forward / backward, cols), the rank-64 merge, the factor operands and the
projection GEMM with a 192-wide adapter segment (K1 = 3 Rp), each against fp64 torch at ranks 33, 48 and 64.  Ranks
below 64 leave zero-padded rank columns, which must stay exactly zero.
Model level: the CUDA path at ranks 48 / 64 against the CPU oracle with the bars of test_parity_gpu.py, the fp32 mode,
the eval merge, exact weight dropout, the CARA_SIDE_TILES=1 routing, the rank-65 refusal and the vit_cp.py entry point."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import cara_oracle as O
from tests.test_kernels_gpu import _gemm_case, _rand_split, _unsplit
from tests.test_parity_gpu import build, check_against, cos, rel, run_step

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANKS = (33, 48, 64)


@pytest.fixture(scope="module")
def K():
    from cara_b200 import kernels
    return kernels


def _pad(t, Rp):
    return torch.nn.functional.pad(t, (0, Rp - t.shape[-1]))


# ------------------------------------------------------------------------------------------------ skinny kernels
@pytest.mark.parametrize("R", RANKS)
@pytest.mark.parametrize("M,Kd", [(50432, 768), (1001, 768), (1001, 3072), (97, 1024)])
def test_rows_fwd_rank64(K, M, Kd, R):
    """T = x A and Uhat = cs (.) T (one slice, as every forward rows pass runs): 64-row CTAs, a ragged last CTA at
    M = 1,001 and 97, rows of every CTA of the 888-CTA grid at M = 50,432."""
    Rp = K.round_rank(R)
    assert Rp == 64
    g = torch.Generator(device="cuda").manual_seed(R)
    x = torch.randn(M, Kd, device="cuda", generator=g).to(BF16)
    A = torch.randn(Kd, R, device="cuda", generator=g) * 0.2
    sc = _pad(torch.randn(1, R, device="cuda", generator=g), Rp).contiguous()
    _, a_t2 = K.factor_operands(A, Rp)
    T, U = K.adapter_rows_fwd(x, a_t2, sc)
    Tref = x.double() @ A.double()
    assert rel(T[:, :R], Tref) < 2e-5
    rows = (T[:, :R].double() - Tref).norm(dim=1) / Tref.norm(dim=1).clamp_min(1e-30)
    assert float(rows.max()) < 1e-4                                  # no row of any CTA is off
    assert rel(_unsplit(U, 1, Rp)[:, :R], Tref * sc[0, :R].double()) < 3e-5
    if R < Rp:
        assert float(T[:, R:].abs().max()) == 0.0
        assert float(U.view(M, 3, Rp)[..., R:].float().abs().max()) == 0.0


@pytest.mark.parametrize("R", RANKS)
@pytest.mark.parametrize("M", [50432, 1001])
@pytest.mark.parametrize("S", [1, 3, 4])
def test_rows_bwd_rank64(K, M, S, R):
    """dU_s = G_s B, dThat = sum_s cs_s (.) dU_s and dcs_s = sum_m dU_s (.) T for 1, 3 (qkv) and 4 (fc1) slices."""
    Rp = K.round_rank(R)
    w = 768
    N = S * w
    g = torch.Generator(device="cuda").manual_seed(100 + R + S)
    G = torch.randn(M, N, device="cuda", generator=g).to(BF16)
    Bf = torch.randn(w, R, device="cuda", generator=g) * 0.2
    sc = _pad(torch.randn(S, R, device="cuda", generator=g), Rp).contiguous()
    T = _pad(torch.randn(M, R, device="cuda", generator=g), Rp).contiguous()
    _, b_t2 = K.factor_operands(Bf, Rp)
    dT, dsc = K.adapter_rows_bwd(G, b_t2, sc, T)
    dU = [G[:, s * w:(s + 1) * w].double() @ Bf.double() for s in range(S)]
    ref = sum(dU[s] * sc[s, :R].double() for s in range(S))
    got = _unsplit(dT, 1, Rp)
    assert rel(got[:, :R], ref) < 3e-5
    rows = (got[:, :R].double() - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-30)
    assert float(rows.max()) < 1e-4
    dsc_ref = torch.stack([(dU[s] * T[:, :R].double()).sum(0) for s in range(S)])
    assert rel(dsc[:, :R], dsc_ref) < 1e-4
    for s in range(S):
        assert rel(dsc[s, :R], dsc_ref[s]) < 1e-4, s
    if R < Rp:
        assert float(got[:, R:].abs().max()) == 0.0 and float(dsc[:, R:].abs().max()) == 0.0


@pytest.mark.parametrize("R", RANKS)
@pytest.mark.parametrize("M,Kc,S", [(50432, 768, 1), (1001, 2304, 3), (50432, 3072, 4), (1001, 1024, 1)])
def test_adapter_cols_rank64(K, M, Kc, S, R):
    """out = sum_s X_s^T (Vhi + Vlo)_s and the column sums of X: 128-column CTAs, two warps per column group."""
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(200 + R)
    X = torch.randn(M, Kc, device="cuda", generator=g).to(BF16)
    vals, V = zip(*[_rand_split((M, R), g) for _ in range(S)])
    V = torch.cat([_pad(v.view(M, 3, R), Rp).view(M, 3 * Rp) for v in V], 1)
    out, cs = K.adapter_cols(X, V, S, Rp, want_colsum=True)
    w = Kc // S
    ref = sum(X[:, s * w:(s + 1) * w].double().t() @ vals[s].double() for s in range(S))
    assert rel(out[:, :R], ref) < 1e-4
    cols = (out[:, :R].double() - ref).norm(dim=0) / ref.norm(dim=0)
    assert float(cols.max()) < 2e-4                                  # every rank column, both warp halves
    assert rel(cs, X.double().sum(0)) < 1e-4
    if R < Rp:
        assert float(out[:, R:].abs().max()) == 0.0


def test_adapter_cols_rank64_hi_only_form():
    """CARA_COLS_HL=1 (contract only the hi block of V) at Rp = 64, in a subprocess since the switch is read once."""
    code = r"""
import torch
from cara_b200 import kernels as K
g = torch.Generator(device="cuda").manual_seed(5)
M, Kc, R = 5001, 2304, 64
X = torch.randn(M, Kc, device="cuda", generator=g).to(torch.bfloat16)
v = torch.randn(M, 3, R, device="cuda", generator=g)
hi = v.to(torch.bfloat16); lo = (v - hi.float()).to(torch.bfloat16)
V = torch.cat([torch.cat([hi[:, s], lo[:, s], hi[:, s]], 1) for s in range(3)], 1)
out, cs = K.adapter_cols(X, V, 3, R, want_colsum=True)
ref = sum(X[:, s * 768:(s + 1) * 768].double().t() @ hi[:, s].double() for s in range(3))
e = float((out.double() - ref).norm() / ref.norm())
ec = float((cs.double() - X.double().sum(0)).norm() / X.double().sum(0).norm())
print("REL", e, ec)
"""
    env = dict(os.environ, PYTHONPATH=ROOT, CARA_COLS_HL="1")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    e, ec = map(float, r.stdout.split("REL")[1].split())
    assert e < 1e-4 and ec < 1e-4, (e, ec)


# ------------------------------------------------------------------------------------------------ merge, operands
@pytest.mark.parametrize("R,S,N,Kd", [(40, 3, 2304, 768), (64, 3, 2304, 768), (64, 1, 768, 3072), (40, 4, 4096, 1024)])
def test_merge_weights_rank64(K, R, S, N, Kd):
    """W + sum_r (Bf (.) cs) A^T with merge_kernel<64>; rank 40 is zero-padded to 64."""
    g = torch.Generator(device="cuda").manual_seed(300 + R)
    W = torch.randn(N, Kd, device="cuda", generator=g) * 0.02
    A = torch.randn(Kd, R, device="cuda", generator=g) * 0.2
    Bf = torch.randn(N // S, R, device="cuda", generator=g) * 0.2
    cs = torch.randn(S, R, device="cuda", generator=g)
    ref = W.double() + torch.cat([(Bf.double() * cs[s].double()) @ A.double().t() for s in range(S)], 0)
    got = K.merge_weights(W, A, Bf, cs).float()
    assert rel(got, ref) < 4e-3                                      # bf16 output rounding
    assert float((got.double() - ref).abs().max()) <= 2.0 ** -8 * float(ref.abs().max())


def test_merge_weights_refuses_rank65(K):
    from cara_b200 import _lib as L
    W = torch.zeros(256, 256, device="cuda")
    with pytest.raises(L.CaraLibraryError, match="64"):
        K.merge_weights(W, torch.zeros(256, 65, device="cuda"), torch.zeros(256, 65, device="cuda"),
                        torch.zeros(1, 65, device="cuda"))


@pytest.mark.parametrize("shape", [(768, 64), (768, 33), (12, 3072, 48), (2, 1280, 64)])
def test_factor_operands_rank64(K, shape):
    """cara_factor_operands at Rp = 64 is bit-identical to the torch formulation."""
    from tests import _torch_ref
    g = torch.Generator().manual_seed(5)
    F = torch.randn(*shape, generator=g) * 0.3
    ext_c, t2_c = _torch_ref.factor_operands(F, 64)
    ext_g, t2_g = K.factor_operands(F.cuda(), 64)
    assert ext_g.shape == ext_c.shape and t2_g.shape == t2_c.shape
    assert torch.equal(ext_g.cpu(), ext_c) and torch.equal(t2_g.cpu(), t2_c)


# ------------------------------------------------------------------------------------------------ GEMM, K1 = 192
@pytest.mark.parametrize("M,N,K0,S,epi,bias", [
    (1001, 768, 3072, 1, 0, True),        # fc2 / proj forward
    (1001, 2304, 768, 3, 0, True),        # qkv
    (1001, 3072, 768, 4, 0, True),
    (1001, 3072, 768, 4, 1, True),        # fc1: GELU epilogue
    (1001, 3072, 768, 1, 1, False),
    (1001, 2304, 768, 3, 1, True),
    (1001, 3072, 768, 1, 2, False),       # fc2 dX: GELU' epilogue
    (1001, 3072, 768, 4, 2, False),
    (1001, 2304, 768, 3, 2, False),
])
def test_gemm_adapter_segment_k1_192(K, M, N, K0, S, epi, bias):
    _gemm_case(K, M, N, K0, 192, S, bias=bias, epi=epi, seed=31)


@pytest.mark.parametrize("N,K0,S,epi,bias", [(3072, 768, 4, 1, True), (2304, 768, 3, 0, True), (768, 3072, 1, 0, True),
                                             (3072, 768, 1, 2, False)])
def test_gemm_adapter_segment_k1_192_bench_size(K, N, K0, S, epi, bias):
    """M = 50,432 (ViT-B/16, batch 256): every persistent CTA and m-tile, checked per 128-row output tile."""
    _gemm_case(K, 50432, N, K0, 192, S, bias=bias, epi=epi, seed=12, blockwise=True)
    torch.cuda.empty_cache()


@pytest.mark.parametrize("B,N,H", [(3, 197, 12), (64, 197, 12), (2, 129, 16)])
def test_gemm_delta_epilogue_k1_192(K, B, N, H):
    """EPI_DELTA with the rank-64 adapter-transpose segment: the output is the plain GEMM's, bit for bit, and delta is
    rowsum(dO (.) (O + O_lo)) per head."""
    from cara_b200 import _lib as L
    g = torch.Generator(device="cuda").manual_seed(41)
    D = 64
    C, M = H * D, B * N
    G = (torch.randn(M, C, device="cuda", generator=g) * 0.5).to(BF16)
    Wt = (torch.randn(C, C, device="cuda", generator=g) * 0.03).to(BF16)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, D ** -0.5)
    a1 = (torch.randn(M, 192, device="cuda", generator=g) * 0.3).to(BF16)
    b1 = (torch.randn(C, 192, device="cuda", generator=g) * 0.1).to(BF16)
    delta = torch.full((B, H, N), float("nan"), device="cuda")
    d_o = K.gemm_cp(G, Wt, a1=a1, b1=b1, epi=L.EPI_DELTA, delta=(o, o_lo, delta, N))
    assert torch.equal(d_o, K.gemm_cp(G, Wt, a1=a1, b1=b1))
    ref_out = G.double() @ Wt.double().t() + a1.double() @ b1.double().t()
    assert rel(d_o, ref_out) < 6e-3
    ref = (d_o.double() * (o.double() + o_lo.double())).view(B, N, H, D).sum(-1).permute(0, 2, 1)
    assert torch.isfinite(delta).all()
    assert float((delta.double() - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))


# ------------------------------------------------------------------------------------------------ model level
@pytest.mark.parametrize("rank", [48, 64])
@pytest.mark.parametrize("geom,batch,scale", [
    (dict(depth=2, num_classes=10), 3, 2.5),                                          # ViT-B width
    (dict(embed_dim=1024, depth=2, num_heads=16, num_classes=100), 2, 1.0),          # ViT-L width
    (dict(embed_dim=1280, depth=2, num_heads=16, patch=14, num_classes=100), 2, 1.0),  # ViT-H/14, D = 80
])
def test_reduced_depth_geometries_rank64_vs_oracle(geom, batch, scale, rank):
    """The bars of test_reduced_depth_geometries_vs_oracle: logits <= 1.5e-2 on a depth-2 model, every gradient
    cosine >= 0.999 and rel-err < 6e-2."""
    g = O.Geometry(rank=rank, **geom)
    vit, st = build(g, scale)
    vit.eval()
    x, y = O.synthetic_batch(g, batch)
    logits, loss, grads = run_step(vit, x, y)
    assert grads["CP_A1"].shape[1] == rank
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, scale)
    e, worst = check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "%s r%d" % (geom, rank),
                             logits_tol=1.5e-2)
    print("r%d %s: logits rel %.3e, worst grad cosine %.6f (%s)" % (rank, geom, e, worst[0], worst[1]))


def test_full_depth_vit_b16_rank64_strict_bar():
    """Full ViT-B/16 at rank 64 against the oracle under the strict bars: logits <= 1e-2, gradient cosine >= 0.999."""
    g = O.Geometry(depth=12, rank=64, num_classes=100)
    vit, st = build(g, 1.0)
    vit.eval()
    x, y = O.synthetic_batch(g, 2)
    logits, loss, grads = run_step(vit, x, y)
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, 1.0)
    e, worst = check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "ViT-B/16 r64 full depth")
    print("ViT-B/16 r64 full depth: logits rel %.3e, worst grad cosine %.6f (%s)" % (e, worst[0], worst[1]))


def test_fp32_mode_rank64_vs_fp64_oracle():
    from cara_b200.fp32 import set_precision
    g = O.Geometry(depth=2, rank=64, num_classes=10)
    vit, st = build(g, 2.5)
    set_precision(vit, "fp32")
    vit.eval()
    x, y = O.synthetic_batch(g, 3)
    logits, loss, grads = run_step(vit, x, y)
    st64 = {k: (v.double() if v.is_floating_point() else v) for k, v in st.items()}
    o_logits, o_loss, o_grads = O.loss_and_grads(st64, g, x.double(), y, 2.5)
    assert rel(logits, o_logits) <= 1e-4
    for k in o_grads:
        assert rel(grads[k], o_grads[k]) <= 1e-3, (k, rel(grads[k], o_grads[k]))


@pytest.mark.parametrize("rank", [40, 64])
def test_eval_merge_rank64_matches_adapter_path_and_oracle(rank):
    """The merged forward (merge_kernel<64>) against the adapter path (<= 1e-2) and both against the oracle's
    materialised merge.  A three-block model gets the reduced-depth bar of test_reduced_depth_geometries_vs_oracle,
    1.5e-2: at rank 64 and scale 2.5 the merged path measured 1.04e-2 on a B200."""
    from cara_b200.merge import merge_cara
    g = O.Geometry(depth=3, rank=rank, num_classes=10)
    vit, st = build(g, 2.5)
    vit.eval()
    x, _ = O.synthetic_batch(g, 4)
    with torch.no_grad():
        y_adapter = vit(x.cuda()).cpu()
        assert merge_cara(vit) == 4 * g.depth
        y_merged = vit(x.cuda()).cpu()
    ref = O.forward_plain(O.merged_weights(st, g, 2.5), g, x)
    e_m, e_a, e_ma = rel(y_merged, ref), rel(y_adapter, ref), rel(y_merged, y_adapter)
    print("r%d eval merge: merged vs oracle %.3e, adapter vs oracle %.3e, merged vs adapter %.3e" % (rank, e_m, e_a, e_ma))
    assert e_m <= 1.5e-2 and e_a <= 1.5e-2
    assert e_ma <= 1e-2


def test_exact_weight_dropout_rank64_replays_through_oracle(monkeypatch):
    """The exact weight-dropout mode at rank 64: the GPU-drawn masks replayed through the oracle's dropout calls."""
    from cara_b200 import wdrop
    g = O.Geometry(depth=2, rank=64, num_classes=10)
    vit, st = build(g, 1.0)
    wdrop.set_weight_dropout(vit, "exact")
    vit.train()
    torch.manual_seed(11)
    torch.cuda.manual_seed_all(11)
    taps = []
    monkeypatch.setattr(wdrop, "MASK_TAP", taps)
    x, y = O.synthetic_batch(g, 3)
    logits, loss, grads = run_step(vit, x, y)
    assert len(taps) == 4 * g.depth
    C = g.embed_dim
    queue = []
    for l in range(g.depth):
        q, p, u, d = [m.cpu() for m in taps[4 * l:4 * l + 4]]
        queue += [q.view(3, C, C).transpose(1, 2), p.t(), u.t(), d.t()]

    def replay(t, p_, train):
        if not train:
            return t
        m = queue.pop(0)
        assert m.shape == t.shape, (m.shape, t.shape)
        return t * m.to(t.dtype)
    monkeypatch.setattr(O, "_wdrop", replay)
    o_logits, o_loss, o_grads = O.loss_and_grads(st, g, x, y, 1.0, train=True, wdrop=0.1)
    assert not queue
    check_against(logits, loss, grads, o_logits, float(o_loss), o_grads, "exact weight dropout r64", logits_tol=1.5e-2)


_ROUTING_CHILD = r"""
import sys, torch
from oracle import cara_oracle as O
from tests.test_parity_gpu import build, run_step
from cara_b200 import kernels as K
g = O.Geometry(depth=2, rank=64, num_classes=10)
vit, _ = build(g, 2.5)
vit.eval()
x, y = O.synthetic_batch(g, 3)
logits, loss, grads = run_step(vit, x, y)
torch.save({"side_tiles": K.side_tiles, "logits": logits, "loss": loss, "grads": grads}, sys.argv[1])
"""


def _routing_run(tmp_path, side_tiles):
    out = os.path.join(str(tmp_path), "side%s.pt" % side_tiles)
    env = dict(os.environ, PYTHONPATH=ROOT, CARA_SIDE_TILES=side_tiles)
    r = subprocess.run([sys.executable, "-c", _ROUTING_CHILD, out], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return torch.load(out)


def test_side_tiles_switch_at_rank64_keeps_the_rows_pass(tmp_path):
    """With CARA_SIDE_TILES=1 an Rp = 64 projection runs the stand-alone rows pass (the GEMM's side tiles cover Rp = 16
    and 32), so the step computes what the default routing computes."""
    a, b = _routing_run(tmp_path, "1"), _routing_run(tmp_path, "0")
    assert a["side_tiles"] and not b["side_tiles"]
    assert torch.equal(a["logits"], b["logits"])                    # the forward has no atomics
    for k in b["grads"]:
        assert cos(a["grads"][k], b["grads"][k]) >= 0.99999 and rel(a["grads"][k], b["grads"][k]) < 1e-4, k


def test_rank65_is_refused_at_the_first_forward():
    g = O.Geometry(depth=1, rank=65, num_classes=10)
    vit, _ = build(g, 1.0)
    x, _ = O.synthetic_batch(g, 1)
    with pytest.raises(NotImplementedError, match="rank > 64"):
        vit(x.cuda())


def test_vit_cp_cli_rank64_trains_saves_and_evaluates(tmp_path):
    """vit_cp.py --dim 64: one epoch of fine-tuning on synthetic data, the checkpoint, and --evaluate of that
    checkpoint (merged with merge_kernel<64>) reproducing the accuracy of the training run."""
    import glob
    env = dict(os.environ, PYTHONPATH=ROOT)
    base = [sys.executable, os.path.join(ROOT, "image_classification", "vit_cp.py"), "--dataset=cifar", "--dim=64",
            "--synthetic"]
    r = subprocess.run(base + ["--epochs=1", "--batch-size=50"], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "e: 0, l:" in r.stdout and "Accuracy:" in r.stdout, r.stdout[-2000:]
    loss = float(r.stdout.split("e: 0, l:")[1].split(",")[0])
    assert 3.0 < loss < 7.0, loss
    ckpts = glob.glob(os.path.join(str(tmp_path), "vit_cifar_*_seed_*.pt"))
    assert len(ckpts) == 1, (ckpts, r.stdout[-2000:])
    assert torch.load(ckpts[0], map_location="cpu")["CP_A1"].shape[1] == 64
    acc_train_run = float(r.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    e = subprocess.run(base + ["--evaluate=" + ckpts[0]], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                       timeout=600)
    assert e.returncode == 0 and "Only evaluation" in e.stdout, e.stderr[-3000:]
    acc_eval = float(e.stdout.strip().splitlines()[-1].split("Accuracy:")[1])
    assert abs(acc_eval - acc_train_run) <= 2.0 / 512 + 1e-9, (acc_eval, acc_train_run)

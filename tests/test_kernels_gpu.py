"""Kernel-level parity (GPU): every C-ABI entry point against a plain fp32 torch statement of the same op
on the same seeded inputs.  bf16 kernels: tolerance is the bf16 rounding of inputs/outputs (rel L2 <= 6e-3);
fp32 kernels: <= 1e-5.  Full-model parity against the CPU oracle lives in test_parity_gpu.py."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


def rel(a, b):
    a = a.double(); b = b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def K():
    from cara_b200 import kernels
    return kernels


def _gemm_case(K, M, N, K0, K1=0, S=1, bias=False, epi=0, seed=0, blockwise=False):
    from cara_b200 import _lib as L
    g = torch.Generator(device="cuda").manual_seed(seed)
    a0 = (torch.randn(M, K0, device="cuda", generator=g) * 0.5).to(BF16)
    b0 = (torch.randn(N, K0, device="cuda", generator=g) * 0.05).to(BF16)
    ref = a0.float() @ b0.float().T
    a1 = b1 = bv = aux = None
    if K1:
        a1 = (torch.randn(M, S * K1, device="cuda", generator=g) * 0.3).to(BF16)
        b1 = (torch.randn(N // S, K1, device="cuda", generator=g) * 0.3).to(BF16)
        w = N // S
        for s in range(S):
            ref[:, s * w:(s + 1) * w] += a1[:, s * K1:(s + 1) * K1].float() @ b1.float().T
    if bias:
        bv = torch.randn(N, device="cuda", generator=g)
        ref += bv
    if epi == L.EPI_DGELU:
        # aux = gelu'(u) as fc1's forward epilogue saved it (bf16); the epilogue multiplies by it
        u = torch.randn(M, N, device="cuda", generator=g).requires_grad_(True)
        torch.nn.functional.gelu(u).sum().backward()
        aux = u.grad.to(BF16)
        ref = ref * aux.float()
        del u
    out = K.gemm_cp(a0, b0, bias=bv, a1=a1, b1=b1, ext_slices=S, epi=epi, aux=aux)
    if epi == L.EPI_GELU:
        # training form: out[0] = gelu'(u) (kept for backward), out[1] = GELU(u), both on the bf16-rounded pre-activation u
        gp, act = out
        u = ref.to(BF16).float().requires_grad_(True)
        act_ref = torch.nn.functional.gelu(u)
        act_ref.sum().backward()
        assert rel(act.float(), act_ref.detach()) < 6e-3, rel(act.float(), act_ref.detach())
        assert rel(gp.float(), u.grad) < 6e-3, rel(gp.float(), u.grad)
        assert float((gp.float() - u.grad).abs().max()) < 2e-2 and float((act.float() - act_ref.detach()).abs().max()) < 5e-2
        if blockwise:
            assert _block_rel(act, act_ref.detach()) < 8e-3 and _block_rel(gp, u.grad) < 8e-3
        # inference form (no derivative output): GELU only
        act2 = K.gemm_cp(a0, b0, bias=bv, a1=a1, b1=b1, ext_slices=S, epi=epi, want_pre=False)[1]
        assert rel(act2.float(), act_ref.detach()) < 6e-3
    else:
        assert rel(out.float(), ref) < 6e-3
        assert not torch.isnan(out.float()).any()
        if blockwise:
            assert _block_rel(out, ref) < 8e-3


def _block_rel(out, ref, bm=128):
    """Worst rel-err over the 128-row output tiles (a single wrong tile among thousands hides in a global norm)."""
    nb = out.shape[0] // bm
    d = (out[:nb * bm].float() - ref[:nb * bm]).view(nb, bm, -1).pow(2).sum((1, 2)).sqrt()
    n = ref[:nb * bm].view(nb, bm, -1).pow(2).sum((1, 2)).sqrt().clamp_min(1e-30)
    return float((d / n).max())


@pytest.mark.parametrize("shape", [
    (128, 256, 64), (128, 256, 768), (591, 768, 768), (1000, 1024, 1024), (257 * 3, 1280, 1280), (4096, 768, 640)])
def test_gemm_plain(K, shape):
    _gemm_case(K, *shape, bias=True)


@pytest.mark.parametrize("M,N,K0,K1,S", [
    (1024, 2304, 768, 16, 3), (1024, 3072, 768, 32, 4), (777, 768, 3072, 16, 1), (394, 3072, 1024, 32, 3),
    (512, 768, 768, 16, 1)])
def test_gemm_adapter_segment(K, M, N, K0, K1, S):
    _gemm_case(K, M, N, K0, K1, S, bias=True)


def test_gemm_epilogues(K):
    from cara_b200 import _lib as L
    _gemm_case(K, 640, 3072, 768, 16, 4, bias=True, epi=L.EPI_GELU)
    _gemm_case(K, 640, 3072, 768, 16, 1, epi=L.EPI_DGELU)


@pytest.mark.parametrize("N,K0,S,epi,bias", [
    (3072, 768, 4, 1, True),      # fc1: GELU epilogue (pre-activation + activation), 4 adapter slices
    (3072, 768, 1, 2, False),     # fc2 dX: GELU' epilogue, adapter-transpose segment
    (2304, 768, 3, 0, True),      # qkv: 3 adapter slices
    (768, 3072, 1, 0, True),      # fc2 (K = 4C)
    (768, 768, 1, 0, True),       # proj
])
def test_gemm_bench_size_epilogues_and_adapter(K, N, K0, S, epi, bias):
    """The measured configuration's GEMMs (BASELINE configs[1]: M = 256 x 197 = 50,432 rows, rank 16 -> K1 = 3 x 16):
    148 persistent CTAs x 394 m-tiles, both TMEM accumulators, every epilogue kind, against fp32 torch -- globally and
    per 128-row output tile."""
    _gemm_case(K, 50432, N, K0, 48, S, bias=bias, epi=epi, seed=11, blockwise=True)
    torch.cuda.empty_cache()


def test_gemm_full_size_linearity(K):
    """c2 size (M = 256*197): linearity f(a+b) = f(a) + f(b) up to bf16 output rounding, and a row checksum."""
    M, N, K0 = 50432, 768, 768
    g = torch.Generator(device="cuda").manual_seed(3)
    a = (torch.randn(M, K0, device="cuda", generator=g)).to(BF16)
    w = (torch.randn(N, K0, device="cuda", generator=g) * 0.03).to(BF16)
    y = K.gemm_cp(a, w).float()
    ref_rowsum = a.float() @ w.float().sum(0)
    assert rel(y.sum(1), ref_rowsum) < 2e-3
    idx = torch.randint(0, M, (512,), device="cuda", generator=g)
    assert rel(y[idx], a[idx].float() @ w.float().T) < 6e-3


@pytest.mark.parametrize("C,act", [(768, BF16), (1024, BF16), (1280, BF16), (256, torch.float32), (768, torch.float32)])
def test_layernorm_fwd_bwd(K, C, act):
    M, rps = 197 * 3 + 5, 197
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(M, C, device="cuda", generator=g) * 2 + 0.3
    delta = torch.randn(M, C, device="cuda", generator=g).to(act)
    rs = torch.rand((M + rps - 1) // rps, device="cuda", generator=g) + 0.5
    gamma = torch.randn(C, device="cuda", generator=g) * 0.1 + 1
    beta = torch.randn(C, device="cuda", generator=g) * 0.1
    rows = torch.arange(M, device="cuda") // rps
    x_ref = (x + rs[rows, None] * delta.float()).requires_grad_(True)
    h_ref = torch.nn.functional.layer_norm(x_ref, (C,), gamma, beta, 1e-6)
    x_out, h, mean, rstd = K.ln_fwd(x, gamma, beta, delta=delta, rowscale=rs, rows_per_sample=rps, act_dtype=act)
    tol = 6e-3 if act == BF16 else 2e-6
    assert rel(x_out, x_ref.detach()) < 1e-6
    assert rel(h.float(), h_ref.detach()) < tol
    dh = torch.randn(M, C, device="cuda", generator=g).to(act)
    dx_in = torch.randn(M, C, device="cuda", generator=g)
    h_ref.backward(dh.float())
    dx, gout = K.ln_bwd(dh, x_out, mean, rstd, gamma, dx_in=dx_in, rowscale=rs, rows_per_sample=rps, want_g=True)
    ref = dx_in + x_ref.grad
    assert rel(dx, ref) < (1e-5 if act == BF16 else 2e-6) * 10
    assert rel(gout.float(), ref * rs[rows, None]) < tol
    # plain LN without residual
    _, h2, _, _ = K.ln_fwd(x, gamma, beta, act_dtype=act)
    assert rel(h2.float(), torch.nn.functional.layer_norm(x, (C,), gamma, beta, 1e-6)) < tol


def _unsplit(U, S, Rp):
    """[M, S*3Rp] (hi|lo|hi) -> fp32 [M, S*Rp] = hi + lo, also checking the duplicated hi block."""
    U = U.float().view(U.shape[0], S, 3, Rp)
    assert torch.equal(U[:, :, 0], U[:, :, 2])
    return (U[:, :, 0] + U[:, :, 1]).reshape(U.shape[0], S * Rp)


def _rand_split(shape, g, scale=1.0):
    """random fp32 tensor and its (hi|lo|hi) bf16 layout along the last dim."""
    v = torch.randn(*shape, device="cuda", generator=g) * scale
    hi = v.to(BF16); lo = (v - hi.float()).to(BF16)
    return hi.float() + lo.float(), torch.cat([hi, lo, hi], -1)


@pytest.mark.parametrize("M,C,R,S", [(197 * 3 + 5, 768, 16, 3), (50432, 768, 16, 4), (1000, 768, 8, 1), (333, 1024, 12, 4)])
def test_layernorm_with_fused_row_contraction(K, M, C, R, S):
    """cara_ln_fwd_rows / cara_ln_bwd_rows = the plain LayerNorm kernels + the stand-alone rows pass on the rows they
    emit: LayerNorm outputs bit-identical, T / Uhat / dThat / dcs equal up to fp32 summation order."""
    rps = 197
    g = torch.Generator(device="cuda").manual_seed(21)
    Rp = K.round_rank(R)
    assert K.ln_rows_fusable(C, Rp) and K.ln_rows_fusable(C, Rp, backward=True)
    x = torch.randn(M, C, device="cuda", generator=g) * 2 + 0.3
    delta = torch.randn(M, C, device="cuda", generator=g).to(BF16)
    rs = torch.rand((M + rps - 1) // rps, device="cuda", generator=g) + 0.5
    gamma = torch.randn(C, device="cuda", generator=g) * 0.1 + 1
    beta = torch.randn(C, device="cuda", generator=g) * 0.1
    A = torch.randn(C, R, device="cuda", generator=g) * 0.1
    _, a_t2 = K.factor_operands(A, Rp)
    cs = torch.nn.functional.pad(torch.randn(S, R, device="cuda", generator=g), (0, Rp - R)).contiguous()
    for with_delta in (True, False):
        kw = dict(delta=delta, rowscale=rs, rows_per_sample=rps) if with_delta else {}
        x0, h0, mean0, rstd0 = K.ln_fwd(x, gamma, beta, act_dtype=BF16, **kw)
        T0, U0 = K.adapter_rows_fwd(h0, a_t2, cs)
        x1, h1, mean1, rstd1, T1, U1 = K.ln_fwd_rows(x, gamma, beta, a_t2, cs, **kw)
        assert torch.equal(h0, h1) and torch.equal(mean0, mean1) and torch.equal(rstd0, rstd1) and torch.equal(x0, x1)
        assert rel(T1, T0) < 2e-6
        assert rel(_unsplit(U1, S, Rp), _unsplit(U0, S, Rp)) < 1e-5
        assert float(T1[:, R:].abs().max()) == 0.0 if R < Rp else True
    _, _, _, _, Tn, Un = K.ln_fwd_rows(x, gamma, beta, a_t2, cs, want_T=False)
    assert Tn is None and torch.equal(Un, U1)
    # backward: g_out is the gradient of a slices = 1 projection with out-side factor B; T = that projection's saved T
    Bf = torch.randn(C, R, device="cuda", generator=g) * 0.1
    _, b_t2 = K.factor_operands(Bf, Rp)
    cs1 = cs[:1].contiguous()
    T = torch.nn.functional.pad(torch.randn(M, R, device="cuda", generator=g), (0, Rp - R)).contiguous()
    dh = torch.randn(M, C, device="cuda", generator=g).to(BF16)
    dx_in = torch.randn(M, C, device="cuda", generator=g)
    for with_in in (True, False):
        kw = dict(dx_in=dx_in if with_in else None, rowscale=rs, rows_per_sample=rps)
        dx0, g0 = K.ln_bwd(dh, x0, mean0, rstd0, gamma, want_g=True, **kw)
        dc1 = torch.zeros(1, Rp, device="cuda")
        dx1, g1, dT1 = K.ln_bwd_rows(dh, x0, mean0, rstd0, gamma, b_t2, cs1, T, dc1, **kw)
        assert rel(dx1, dx0) < 1e-6 and rel(g1.float(), g0.float()) < 1e-3   # two compilations of the same formulas
        dT0, dc0 = K.adapter_rows_bwd(g1, b_t2, cs1, T)                       # the stand-alone pass on the same G
        assert rel(_unsplit(dT1, 1, Rp), _unsplit(dT0, 1, Rp)) < 1e-5
        assert rel(dc1, dc0) < 1e-4



@pytest.mark.parametrize("M,Kd,R,S", [(1000, 768, 16, 3), (50432, 768, 16, 4), (333, 3072, 8, 1), (700, 1024, 32, 4)])
def test_adapter_rows_fwd(K, M, Kd, R, S):
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(M, Kd, device="cuda", generator=g).to(BF16)
    A = torch.randn(Kd, R, device="cuda", generator=g) * 0.2
    sc = torch.zeros(S, Rp, device="cuda"); sc[:, :R] = torch.randn(S, R, device="cuda", generator=g)
    _, a_t2 = K.factor_operands(A, Rp)
    T, U = K.adapter_rows_fwd(x, a_t2, sc)
    Tref = torch.nn.functional.pad(x.double() @ A.double(), (0, Rp - R)).float()
    assert rel(T, Tref) < 2e-5          # factor carried as hi+lo: far below the 2e-3 of a single bf16
    Uref = torch.cat([Tref * sc[s] for s in range(S)], 1)
    assert rel(_unsplit(U, S, Rp), Uref) < 3e-5
    if R < Rp:
        assert float(U.view(M, S, 3, Rp)[..., R:].float().abs().max()) == 0.0


@pytest.mark.parametrize("M,N,R,S", [(1000, 2304, 16, 3), (50432, 768, 16, 1), (515, 3072, 8, 4), (700, 4096, 32, 4)])
def test_adapter_rows_bwd(K, M, N, R, S):
    Rp = K.round_rank(R)
    w = N // S
    g = torch.Generator(device="cuda").manual_seed(4)
    G = torch.randn(M, N, device="cuda", generator=g).to(BF16)
    Bf = torch.randn(w, R, device="cuda", generator=g) * 0.2
    sc = torch.zeros(S, Rp, device="cuda"); sc[:, :R] = torch.randn(S, R, device="cuda", generator=g)
    T = torch.randn(M, Rp, device="cuda", generator=g)
    _, b_t2 = K.factor_operands(Bf, Rp)
    dT, dsc = K.adapter_rows_bwd(G, b_t2, sc, T)
    dU = [torch.nn.functional.pad(G[:, s * w:(s + 1) * w].double() @ Bf.double(), (0, Rp - R)).float() for s in range(S)]
    assert rel(_unsplit(dT, 1, Rp), sum(dU[s] * sc[s] for s in range(S))) < 3e-5
    assert rel(dsc, torch.stack([(dU[s] * T).sum(0) for s in range(S)])) < 1e-4


@pytest.mark.parametrize("M,Kc,R,S", [(1000, 768, 16, 1), (50432, 2304, 16, 3), (515, 3072, 8, 4), (700, 1024, 32, 1),
                                      (50432, 3072, 16, 1)])
def test_adapter_cols(K, M, Kc, R, S):
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(M, Kc, device="cuda", generator=g).to(BF16)
    vals, V = zip(*[_rand_split((M, Rp), g) for _ in range(S)])
    V = torch.cat(V, 1)
    out, cs = K.adapter_cols(X, V, S, Rp, want_colsum=True)
    w = Kc // S
    ref = sum(X[:, s * w:(s + 1) * w].double().t() @ vals[s].double() for s in range(S)).float()
    assert rel(out, ref) < 1e-4
    assert rel(cs, X.float().sum(0)) < 1e-4


@pytest.mark.parametrize("M,N,K0,R,S,epi", [
    (1000, 768, 768, 16, 1, 0), (777, 2304, 768, 8, 3, 0), (640, 3072, 1024, 32, 4, 0), (515, 1024, 4096, 32, 1, 0),
    (128, 256, 64, 16, 1, 0),                                   # a single panel, a single k-block
    (50432, 2304, 768, 16, 3, 0), (50432, 768, 768, 16, 1, 0), (50432, 768, 3072, 16, 1, 0)])   # the bench shapes
def test_gemm_side_tiles_forward(K, M, N, K0, R, S, epi):
    """The fused projection with its side tiles: ONE launch computes T = x A, Uhat_s = cs_s (.) T (side tiles) and
    y = x W^T + b + Uhat B^T (output tiles reading the side tiles' rows behind the per-panel flags).  Checked against
    fp64 torch for T / Uhat and fp32 torch for y -- twice in a row (the generation counter must advance)."""
    from cara_b200 import _lib as L
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(21)
    x = (torch.randn(M, K0, device="cuda", generator=g) * 0.5).to(BF16)
    W = (torch.randn(N, K0, device="cuda", generator=g) * 0.05).to(BF16)
    bias = torch.randn(N, device="cuda", generator=g)
    A = torch.randn(K0, R, device="cuda", generator=g) * 0.1
    Bf = torch.randn(N // S, R, device="cuda", generator=g) * 0.2
    cs = torch.zeros(S, Rp, device="cuda"); cs[:, :R] = torch.randn(S, R, device="cuda", generator=g)
    _, a_t2 = K.factor_operands(A, Rp)
    b_ext, _ = K.factor_operands(Bf, Rp)
    Tref = torch.nn.functional.pad(x.double() @ A.double(), (0, Rp - R)).float()
    Uref = torch.cat([Tref * cs[s] for s in range(S)], 1)
    w = N // S
    ref = x.float() @ W.float().T + bias
    for s in range(S):
        ref[:, s * w:(s + 1) * w] += (Tref[:, :R] * cs[s, :R]) @ Bf.T
    for _ in range(2):
        T = torch.full((M, Rp), float("nan"), device="cuda")
        U = torch.full((M, S * 3 * Rp), float("nan"), device="cuda", dtype=BF16)
        side = K.Side(L.SIDE_FWD, a_t2, cs, T, U)
        out = K.gemm_cp(x, W, bias=bias, a1=U, b1=b_ext, ext_slices=S, epi=epi, side=side)
        assert rel(T, Tref) < 2e-5
        assert rel(_unsplit(U, S, Rp), Uref) < 3e-5
        if epi == L.EPI_GELU:
            act_ref = torch.nn.functional.gelu(ref.to(BF16).float())
            assert rel(out[1].float(), act_ref) < 6e-3 and _block_rel(out[1], act_ref) < 8e-3
        else:
            assert rel(out.float(), ref) < 6e-3 and _block_rel(out, ref) < 8e-3
    del ref
    torch.cuda.empty_cache()


@pytest.mark.parametrize("M,N,K0,R,S,epi", [
    (1000, 768, 768, 16, 1, 0), (777, 768, 2304, 8, 3, 0), (640, 1024, 4096, 32, 4, 0), (515, 3072, 768, 16, 1, 0),
    (50432, 768, 2304, 16, 3, 0), (50432, 768, 3072, 16, 4, 0), (50432, 768, 768, 16, 1, 0)])   # qkv / fc1 / proj dX
def test_gemm_side_tiles_backward(K, M, N, K0, R, S, epi):
    """The dX GEMM with its side tiles (G = dY [M, K0] against W^T stored [N, K0]): dU_s = G_s B per K-slice,
    dThat = sum_s cs_s (.) dU_s feeds the adapter-transpose segment, dcs_s = sum_m dU_s (.) T is accumulated."""
    from cara_b200 import _lib as L
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(22)
    G = (torch.randn(M, K0, device="cuda", generator=g) * 0.5).to(BF16)
    Wt = (torch.randn(N, K0, device="cuda", generator=g) * 0.05).to(BF16)
    wk = K0 // S
    Bf = torch.randn(wk, R, device="cuda", generator=g) * 0.1          # out-side factor (per K-slice of G)
    A = torch.randn(N, R, device="cuda", generator=g) * 0.2            # in-side factor: dX += dThat A^T
    cs = torch.zeros(S, Rp, device="cuda"); cs[:, :R] = torch.randn(S, R, device="cuda", generator=g)
    T = torch.randn(M, Rp, device="cuda", generator=g)
    _, b_t2 = K.factor_operands(Bf, Rp)
    a_ext, _ = K.factor_operands(A, Rp)
    aux = (torch.rand(M, N, device="cuda", generator=g) * 1.3 - 0.15).to(BF16) if epi == L.EPI_DGELU else None   # a gelu'(u)
    dU = [torch.nn.functional.pad(G[:, s * wk:(s + 1) * wk].double() @ Bf.double(), (0, Rp - R)).float() for s in range(S)]
    dTref = sum(dU[s] * cs[s] for s in range(S))
    ref = G.float() @ Wt.float().T + dTref[:, :R] @ A.T
    if aux is not None:
        ref = ref * aux.float()
    dcs_ref = torch.stack([(dU[s] * T).sum(0) for s in range(S)])
    dcs = torch.zeros(S, Rp, device="cuda")
    for rep_ in range(2):
        dT = torch.full((M, 3 * Rp), float("nan"), device="cuda", dtype=BF16)
        side = K.Side(L.SIDE_BWD, b_t2, cs, T, dT, dcs)
        dx = K.gemm_cp(G, Wt, a1=dT, b1=a_ext, ext_slices=1, epi=epi, aux=aux, side=side)
        assert rel(_unsplit(dT, 1, Rp), dTref) < 3e-5
        assert rel(dx.float(), ref) < 6e-3 and _block_rel(dx, ref) < 8e-3
        assert rel(dcs, (rep_ + 1) * dcs_ref) < 1e-4               # accumulated, not overwritten
    del ref
    torch.cuda.empty_cache()


def test_gemm_adapter_segment_split_precision(K):
    """End to end through the split operands: x A diag(c) B^T added by the GEMM's adapter segment is accurate
    to ~1e-4 relative (a single-bf16 chain would sit at ~3e-3)."""
    M, Kd, N, R, S = 1024, 768, 2304, 16, 3
    Rp = K.round_rank(R)
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(M, Kd, device="cuda", generator=g).to(BF16)
    A = torch.randn(Kd, R, device="cuda", generator=g) * 0.2
    Bf = torch.randn(N // S, R, device="cuda", generator=g) * 0.2
    cs = torch.randn(S, R, device="cuda", generator=g)
    _, a_t2 = K.factor_operands(A, Rp)
    b_ext, _ = K.factor_operands(Bf, Rp)
    T, U = K.adapter_rows_fwd(x, a_t2, torch.nn.functional.pad(cs, (0, Rp - R)).contiguous())
    zero_w = torch.zeros(N, Kd, device="cuda", dtype=BF16)
    big = 64.0   # keep the bf16 output rounding out of the way: compare the fp32-accurate part via a scaled copy
    y = K.gemm_cp(x, zero_w, a1=U, b1=b_ext, ext_slices=S).float()
    ref = torch.cat([((x.double() @ A.double()) * cs[s].double()) @ Bf.double().t() for s in range(S)], 1).float()
    assert rel(y, ref) < 3e-3            # bf16 output rounding only
    assert abs(float((y - ref).mean())) < 1e-4 * float(ref.abs().mean()) + 1e-6


@pytest.mark.parametrize("B,N,H,D", [(3, 197, 12, 64), (2, 257, 16, 80), (2, 64, 4, 64), (1, 50, 2, 64), (2, 17, 3, 64),
                                     (1, 128, 2, 80),
                                     (40, 197, 12, 64),     # 480 heads: every persistent CTA walks over 3-4 heads
                                     (80, 256, 4, 64)])     # N = 256: single Q/K pair (no prefetch), 2+ heads per CTA
def test_attention_fwd_bwd(K, B, N, H, D):
    g = torch.Generator(device="cuda").manual_seed(6)
    C = H * D
    qkv = (torch.randn(B, N, 3, H, D, device="cuda", generator=g) * 1.0).to(BF16)
    scale = D ** -0.5
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale)
    q, k, v = [t.float().requires_grad_(True) for t in qkv.permute(2, 0, 3, 1, 4)]
    att = ((q @ k.transpose(-2, -1)) * scale).softmax(-1)
    oref = (att @ v).transpose(1, 2).reshape(B * N, C)
    assert rel(o.float(), oref.detach()) < 6e-3
    assert rel(o.float() + o_lo.float(), oref.detach()) < 3e-3      # (hi, lo) pair: only P's bf16 rounding is left
    o_inf, no_lo, no_lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale, train=False)
    assert no_lo is None and no_lse is None and torch.equal(o_inf, o)
    lref = torch.logsumexp((q @ k.transpose(-2, -1)) * scale, -1) / math.log(2.0)
    assert rel(lse, lref.detach()) < 1e-4
    d_o = torch.randn(B * N, C, device="cuda", generator=g).to(BF16)
    oref.backward(d_o.float())
    dqkv = K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, scale).view(B, N, 3, H, D)
    dref = torch.stack([q.grad, k.grad, v.grad], 0).permute(1, 3, 0, 2, 4)
    for i, name in enumerate("qkv"):
        assert rel(dqkv[:, :, i].float(), dref[:, :, i]) < 1.2e-2, name


@pytest.mark.parametrize("B,N,H,R", [(3, 197, 12, 16), (256, 197, 12, 16), (5, 50, 4, 0), (2, 256, 16, 32),
                                     (2, 129, 12, 16),      # a second query tile of one row
                                     (3, 209, 12, 16)])     # N = 209: the backward without the Q/K prefetch
def test_gemm_delta_epilogue_feeds_attention_backward(K, B, N, H, R):
    """EPI_DELTA: the output projection's dX GEMM (frozen W^T + adapter-transpose segment) also writes
    delta[b,h,n] = sum_d bf16(dO) (O_hi + O_lo) -- bit-for-bit the dO it stores, so it must equal the stand-alone
    pre-pass of cara_attn_bwd to fp32 summation order, and the attention backward fed with it must equal the
    backward that runs its own pre-pass (autograd of cara.py:44-58)."""
    from cara_b200 import _lib as L
    g = torch.Generator(device="cuda").manual_seed(11)
    D = 64
    C, M = H * D, B * N
    G = (torch.randn(M, C, device="cuda", generator=g) * 0.5).to(BF16)
    Wt = (torch.randn(C, C, device="cuda", generator=g) * 0.03).to(BF16)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g).to(BF16)
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, D ** -0.5)
    a1 = b1 = None
    if R:
        a1 = (torch.randn(M, 3 * R, device="cuda", generator=g) * 0.3).to(BF16)
        b1 = (torch.randn(C, 3 * R, device="cuda", generator=g) * 0.1).to(BF16)
    delta = torch.full((B, H, N), float("nan"), device="cuda")
    d_o = K.gemm_cp(G, Wt, a1=a1, b1=b1, epi=L.EPI_DELTA, delta=(o, o_lo, delta, N))
    plain = K.gemm_cp(G, Wt, a1=a1, b1=b1)
    assert torch.equal(d_o, plain)                                  # the extra epilogue work never touches the output
    ref = (d_o.float() * (o.float() + o_lo.float())).view(B, N, H, D).sum(-1).permute(0, 2, 1)
    assert torch.isfinite(delta).all()
    assert float((delta - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    mine = K.attn_bwd(qkv.view(-1), None, None, lse, d_o, B, N, H, D, D ** -0.5, delta=delta)
    theirs = K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, D ** -0.5)
    assert rel(mine.float(), theirs.float()) < 1e-3                # fp32 summation order of delta -> a few bf16 roundings flip


def test_patch_embed_path(K):
    B, S, P, C = 3, 224, 16, 768
    g = torch.Generator(device="cuda").manual_seed(7)
    img = torch.randn(B, 3, S, S, device="cuda", generator=g)
    Wc = torch.randn(C, 3, P, P, device="cuda", generator=g) * 0.03
    bc = torch.randn(C, device="cuda", generator=g) * 0.1
    cls = torch.randn(C, device="cuda", generator=g); pos = torch.randn(197, C, device="cuda", generator=g)
    patches = K.patchify(img, P, 768)
    pe = K.gemm_cp(patches, Wc.reshape(C, -1).to(BF16).contiguous(), bias=bc)
    x = K.assemble_tokens(pe, cls, pos, B, 197, C)
    ref = torch.nn.functional.conv2d(img, Wc, bc, stride=P).flatten(2).transpose(1, 2)
    ref = torch.cat([cls.expand(B, 1, C), ref], 1) + pos
    assert rel(x.view(B, 197, C), ref) < 6e-3
    # ViT-H/14 geometry: K = 588 zero padded to 640
    patches = K.patchify(img, 14, 640)
    ref = torch.nn.functional.unfold(img, 14, stride=14).transpose(1, 2).reshape(-1, 588)
    assert rel(patches[:, :588].float(), ref) < 6e-3 and float(patches[:, 588:].float().abs().max()) == 0.0


def test_merge_adamw_sgemm(K):
    g = torch.Generator(device="cuda").manual_seed(8)
    N, Kd, R, S = 2304, 768, 16, 3
    W = torch.randn(N, Kd, device="cuda", generator=g) * 0.02
    A = torch.randn(Kd, R, device="cuda", generator=g) * 0.2
    Bf = torch.randn(N // S, R, device="cuda", generator=g) * 0.2
    cs = torch.randn(S, R, device="cuda", generator=g)
    ref = W + torch.cat([(Bf * cs[s]) @ A.t() for s in range(S)], 0)
    assert rel(K.merge_weights(W, A, Bf, cs).float(), ref) < 4e-3
    p = torch.randn(12345, device="cuda", generator=g); pr = torch.nn.Parameter(p.clone())
    opt = torch.optim.AdamW([pr], lr=1e-3, weight_decay=1e-4)
    m = torch.zeros_like(p); v = torch.zeros_like(p)
    for step in range(1, 4):
        gr = torch.randn(12345, device="cuda", generator=g)
        pr.grad = gr.clone(); opt.step()
        K.adamw_step(p, gr, m, v, 1e-3, step)
        assert rel(p, pr.detach()) < 1e-6
    a = torch.randn(77, 130, device="cuda", generator=g); b = torch.randn(100, 130, device="cuda", generator=g)
    bias = torch.randn(100, device="cuda", generator=g)
    assert rel(K.sgemm(a, b.t(), bias=bias), a @ b.t() + bias) < 1e-5
    assert rel(K.sgemm(a.t(), a), a.t() @ a) < 1e-5


@pytest.mark.parametrize("B,N,H,D", [(2, 197, 3, 64), (1, 257, 2, 80), (2, 33, 2, 64), (1, 288, 2, 64), (3, 32, 2, 80)])
def test_fp32_mode_attention_and_gelu(K, B, N, H, D):
    g = torch.Generator(device="cuda").manual_seed(11)
    qkv = torch.randn(B, N, 3, H, D, device="cuda", generator=g)
    scale = D ** -0.5
    o, lse = K.attn_f32_fwd(qkv.view(-1), B, N, H, D, scale)
    q, k, v = [t.double().requires_grad_(True) for t in qkv.permute(2, 0, 3, 1, 4)]
    att = ((q @ k.transpose(-2, -1)) * scale).softmax(-1)
    oref = (att @ v).transpose(1, 2).reshape(B * N, H * D)
    assert rel(o, oref.detach()) < 2e-6
    d_o = torch.randn(B * N, H * D, device="cuda", generator=g)
    oref.backward(d_o.double())
    dqkv = K.attn_f32_bwd(qkv.view(-1), o, lse, d_o, B, N, H, D, scale).view(B, N, 3, H, D)
    dref = torch.stack([q.grad, k.grad, v.grad], 0).permute(1, 3, 0, 2, 4)
    assert rel(dqkv, dref) < 5e-6
    u = torch.randn(1000, 37, device="cuda", generator=g) * 2
    ud = u.double().requires_grad_(True)
    yd = torch.nn.functional.gelu(ud)
    assert rel(K.gelu_f32(u), yd.detach()) < 1e-6
    dy = torch.randn_like(u)
    yd.backward(dy.double())
    assert rel(K.gelu_f32(u, dy=dy), ud.grad) < 2e-6


@pytest.mark.parametrize("shape,Rp", [((768, 16), 16), ((768, 8), 16), ((12, 3072, 16), 16), ((2, 1024, 20), 32), ((5, 7), 16)])
def test_factor_operands_kernel_matches_torch_formulation(K, shape, Rp):
    """cara_factor_operands (pad + bf16 hi/lo split + both operand layouts in one launch) is bit-identical to the
    torch formulation the host-side staging tests use."""
    g = torch.Generator().manual_seed(5)
    F = torch.randn(*shape, generator=g) * 0.3
    from tests import _torch_ref
    ext_c, t2_c = _torch_ref.factor_operands(F, Rp)        # torch formulation on the CPU
    ext_g, t2_g = K.factor_operands(F.cuda(), Rp)          # CUDA tensors -> the kernel
    assert ext_g.shape == ext_c.shape and t2_g.shape == t2_c.shape
    assert torch.equal(ext_g.cpu(), ext_c) and torch.equal(t2_g.cpu(), t2_c)

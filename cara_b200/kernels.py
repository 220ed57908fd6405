"""Tensor-level wrappers over the C ABI (one function per entry point of include/cara_b200.h).

PyTorch owns the memory and the stream; these functions only pass ``data_ptr()``s, sizes and
``torch.cuda.current_stream()`` through ctypes.  Every function requires CUDA tensors: there is no CPU
path here by design.
"""
import ctypes as C
import os

import torch

from . import _lib as L

BF16, F32 = torch.bfloat16, torch.float32
launch_count = 0  # number of cara_* kernel launches issued (bench.py reports it as gpu_launches)
param_generation = 0  # bumped by adamw_step: parameters changed behind autograd's version counters
# CARA_SIDE_TILES=1: compute the rank-R row contractions (T = x A, dU = g B) as side tiles inside the projection GEMM's
# launch instead of the stand-alone rows kernel.  Opt-in: correct (tests/test_kernels_gpu.py::test_gemm_side_tiles_*)
# and step-neutral on B200 (profiles/r02_side_tiles.md); with the LayerNorm fusion below no stand-alone rows pass is left.
side_tiles = os.environ.get("CARA_SIDE_TILES", "0") == "1"
# the attention backward's rowsum(dO (.) O) out of the output projection's dX GEMM epilogue (CARA_DELTA_IN_GEMM=0: the
# stand-alone pre-pass inside cara_attn_bwd)
delta_in_gemm = os.environ.get("CARA_DELTA_IN_GEMM", "1") == "1"
gemm_events = None  # bench.py: list of (start event, end event, algorithmic flops) per fused-projection launch
_dev = [None]


def _prep(t):
    global launch_count
    if not t.is_cuda:
        raise L.CaraLibraryError("cara_b200 kernels need CUDA tensors (no CPU fallback)")
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if _dev[0] != idx:
        L.check(L.lib().cara_set_device(idx), "cara_set_device")
        _dev[0] = idx
    launch_count += 1
    return torch.cuda.current_stream(t.device).cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


MAX_RANK = 64   # the largest rank the rank-R kernels (skinny, merge) are instantiated for


def round_rank(r):
    """The padded rank Rp (16, 32 or 64) the bf16 kernels run a rank-r adapter at."""
    if r > MAX_RANK:
        raise ValueError("rank %d > %d is not supported by the bf16 kernels" % (r, MAX_RANK))
    return 16 if r <= 16 else 32 if r <= 32 else 64


_sync_ws = {}


def sync_workspace(device):
    """The 16 KB of zero-initialised device words (generation counter + one flag per 128-row panel) the GEMM's side
    tiles synchronise through; one per device, lent to every call (see include/cara_b200.h, sync_ws)."""
    ws = _sync_ws.get(device)
    if ws is None:
        ws = _sync_ws[device] = torch.zeros(L.SYNC_WORDS, device=device, dtype=torch.int32)
    return ws


class Side:
    """Side tiles of one fused projection (see cara_gemm_cp): the rank-R row contraction of the GEMM's own A0 rows.
    ``mode`` L.SIDE_FWD: T = a0 P^T, Uhat = split(scales (.) T) -> ``U`` (the GEMM's a1), ``T`` saved (or None).
    ``mode`` L.SIDE_BWD: dThat = split(sum_s scales[s] (.) (a0_s P^T)) -> ``U``, ``dc`` += sum_m dU_s (.) T."""
    __slots__ = ("mode", "P", "scales", "T", "U", "dc")

    def __init__(self, mode, P, scales, T, U, dc=None):
        self.mode, self.P, self.scales, self.T, self.U, self.dc = mode, P, scales, T, U, dc


def _fill_side(d, side, M, K0, device):
    S, Rp = side.scales.shape
    kslices = S if side.mode == L.SIDE_BWD else 1
    assert side.P.dtype == BF16 and side.P.shape == (2 * Rp, K0 // kslices) and side.P.stride(1) == 1
    assert side.scales.dtype == F32 and side.scales.is_contiguous()
    assert side.U.dtype == BF16 and side.U.shape[0] == M and side.U.stride(1) == 1
    assert side.U.shape[1] == (3 * Rp if side.mode == L.SIDE_BWD else S * 3 * Rp)
    if side.T is not None:
        assert side.T.dtype == F32 and side.T.shape == (M, Rp) and side.T.is_contiguous()
    d.side, d.side_rp, d.side_slices = side.mode, Rp, S
    d.P, d.ldp = side.P.data_ptr(), side.P.stride(0)
    d.side_scales, d.side_T = side.scales.data_ptr(), _p(side.T)
    d.side_U, d.side_ldu = side.U.data_ptr(), side.U.stride(0)
    d.side_dc = _p(side.dc)
    d.sync_ws = sync_workspace(device).data_ptr()


def gemm_cp(a0, b0, bias=None, a1=None, b1=None, ext_slices=1, epi=L.EPI_NONE, out=None, out2=None, aux=None,
            want_pre=True, num_sms=0, side=None, delta=None):
    """out[M,N] = a0[M,K0] b0[N,K0]^T + bias (+ adapter segment a1/b1), see cara_gemm_cp.  ``side`` (a ``Side``):
    the kernel also computes the low-rank operand -- then ``a1`` must be ``side.U``, which it fills before use.
    ``delta`` = (o, o_lo, delta_out [B,H,N] fp32, seq_n) with epi = EPI_DELTA: the attention backward's row term."""
    st = _prep(a0)
    M, K0 = a0.shape
    N = b0.shape[0]
    assert a0.dtype == BF16 and b0.dtype == BF16 and b0.shape[1] == K0
    assert a0.stride(1) == 1 and b0.stride(1) == 1
    d = L.GemmDesc()
    d.M, d.N, d.K0 = M, N, K0
    d.A0, d.lda0, d.B0, d.ldb0 = a0.data_ptr(), a0.stride(0), b0.data_ptr(), b0.stride(0)
    if a1 is not None:
        K1 = b1.shape[1]
        assert a1.dtype == BF16 and b1.dtype == BF16 and a1.shape == (M, ext_slices * K1)
        assert b1.shape[0] * ext_slices == N and a1.stride(1) == 1 and b1.stride(1) == 1
        d.K1, d.ext_slices = K1, ext_slices
        d.A1, d.lda1, d.B1, d.ldb1 = a1.data_ptr(), a1.stride(0), b1.data_ptr(), b1.stride(0)
    if side is not None:
        assert a1 is not None and a1.data_ptr() == side.U.data_ptr()
        _fill_side(d, side, M, K0, a0.device)
    if bias is not None:
        assert bias.dtype == F32 and bias.numel() == N and bias.is_contiguous()
        d.bias = bias.data_ptr()
    if out is None and (epi != L.EPI_GELU or want_pre):
        out = torch.empty((M, N), device=a0.device, dtype=BF16)
    if out is not None:
        d.out, d.ldo = out.data_ptr(), out.stride(0)
    if epi == L.EPI_GELU:
        if out2 is None:
            out2 = torch.empty((M, N), device=a0.device, dtype=BF16)
        d.out2, d.ldo2 = out2.data_ptr(), out2.stride(0)
    if epi == L.EPI_DGELU:
        assert aux is not None and aux.dtype == BF16 and aux.shape == (M, N)
        d.aux, d.ldaux = aux.data_ptr(), aux.stride(0)
    if epi == L.EPI_DELTA:
        o_hi, o_lo, dl, seq_n = delta
        assert o_hi.dtype == BF16 and o_lo.dtype == BF16 and o_hi.shape == (M, N) and o_lo.shape == (M, N)
        assert dl.dtype == F32 and dl.is_contiguous() and dl.numel() == M * (N // 64) and M % seq_n == 0
        d.aux, d.ldaux, d.aux2, d.ldaux2 = o_hi.data_ptr(), o_hi.stride(0), o_lo.data_ptr(), o_lo.stride(0)
        d.delta, d.seq_n = dl.data_ptr(), seq_n
    d.epi, d.num_sms = epi, num_sms
    if gemm_events is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(L.lib().cara_gemm_cp(C.byref(d), st), "cara_gemm_cp")
        e1.record()
        Rp = d.side_rp if side is not None else 0
        # algorithmic flops: frozen product + adapter segment (rank Rp) + the side contraction (rank Rp)
        gemm_events.append((e0, e1, 2.0 * M * N * (K0 + (d.K1 // 3 if a1 is not None else 0)) + 2.0 * M * K0 * Rp))
    else:
        L.check(L.lib().cara_gemm_cp(C.byref(d), st), "cara_gemm_cp")
    return (out, out2) if epi == L.EPI_GELU else out


def ln_fwd(x, gamma, beta, delta=None, rowscale=None, rows_per_sample=1, eps=1e-6, act_dtype=BF16,
           write_x=True, want_stats=True):
    """Returns (x_out, h, mean, rstd).  x fp32 [M,C]; x_out aliases x when delta is None."""
    st = _prep(x)
    M, Cc = x.shape
    assert x.dtype == F32 and x.is_contiguous()
    if delta is not None:
        assert delta.shape == x.shape and delta.dtype == act_dtype and delta.is_contiguous()
    x_out = torch.empty_like(x) if (delta is not None and write_x) else (x if delta is None else None)
    h = torch.empty((M, Cc), device=x.device, dtype=act_dtype)
    mean = torch.empty(M, device=x.device, dtype=F32) if want_stats else None
    rstd = torch.empty(M, device=x.device, dtype=F32) if want_stats else None
    L.check(L.lib().cara_ln_fwd(x.data_ptr(), _p(delta), _p(rowscale), rows_per_sample,
                                _p(x_out) if delta is not None else None, gamma.data_ptr(), beta.data_ptr(),
                                h.data_ptr(), _p(mean), _p(rstd), M, Cc, eps, int(act_dtype == F32), st), "cara_ln_fwd")
    return x_out, h, mean, rstd


def ln_bwd(dh, x, mean, rstd, gamma, dx_in=None, rowscale=None, rows_per_sample=1, want_g=False):
    """Returns (dx_out fp32, g_out or None)."""
    st = _prep(x)
    M, Cc = x.shape
    dx_out = torch.empty_like(x)
    g_out = torch.empty((M, Cc), device=x.device, dtype=dh.dtype) if want_g else None
    L.check(L.lib().cara_ln_bwd(dh.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
                                _p(dx_in), dx_out.data_ptr(), _p(g_out), _p(rowscale), rows_per_sample, M, Cc,
                                int(dh.dtype == F32), st), "cara_ln_bwd")
    return dx_out, g_out


# the K = C row contractions inside the LayerNorm kernels that produce their operand (csrc/ln_rows.cu).
# CARA_LN_ROWS: bit 0 = forward (T = h A for qkv / fc1), bit 1 = backward (dU = G B for proj / fc2); 0 = stand-alone passes
ln_rows = int(os.environ.get("CARA_LN_ROWS", "3"))


def ln_rows_fusable(Cc, Rp, backward=False):
    return bool(ln_rows & (2 if backward else 1)) and bool(L.lib().cara_ln_rows_supported(int(Cc), int(Rp)))


def ln_fwd_rows(x, gamma, beta, a_t2, scales, delta=None, rowscale=None, rows_per_sample=1, eps=1e-6, want_T=True):
    """``ln_fwd`` (bf16 activations) that also contracts the rows it emits with the consumer's in-side factor:
    returns (x_out, h, mean, rstd, T fp32 [M,Rp] or None, Uhat bf16 [M,S*3Rp]) -- see cara_ln_fwd_rows."""
    st = _prep(x)
    M, Cc = x.shape
    S, Rp = scales.shape
    assert x.dtype == F32 and x.is_contiguous() and a_t2.shape == (2 * Rp, Cc) and a_t2.is_contiguous()
    assert scales.dtype == F32 and scales.is_contiguous()
    if delta is not None:
        assert delta.shape == x.shape and delta.dtype == BF16 and delta.is_contiguous()
    x_out = torch.empty_like(x) if delta is not None else x
    h = torch.empty((M, Cc), device=x.device, dtype=BF16)
    mean = torch.empty(M, device=x.device, dtype=F32)
    rstd = torch.empty(M, device=x.device, dtype=F32)
    T = torch.empty((M, Rp), device=x.device, dtype=F32) if want_T else None
    U = torch.empty((M, S * 3 * Rp), device=x.device, dtype=BF16)
    L.check(L.lib().cara_ln_fwd_rows(x.data_ptr(), _p(delta), _p(rowscale), rows_per_sample,
                                     _p(x_out) if delta is not None else None, gamma.data_ptr(), beta.data_ptr(),
                                     h.data_ptr(), mean.data_ptr(), rstd.data_ptr(), M, Cc, eps, a_t2.data_ptr(),
                                     scales.data_ptr(), S, Rp, _p(T), U.data_ptr(), st), "cara_ln_fwd_rows")
    return x_out, h, mean, rstd, T, U


def ln_bwd_rows(dh, x, mean, rstd, gamma, b_t2, scales, T, dsc, dx_in=None, rowscale=None, rows_per_sample=1):
    """``ln_bwd`` with g_out that also contracts g_out with the out-side factor of the projection it is the gradient
    of: returns (dx_out, g_out, dThat bf16 [M,3Rp]); dsc fp32 [1,Rp] is accumulated into -- see cara_ln_bwd_rows."""
    st = _prep(x)
    M, Cc = x.shape
    S, Rp = scales.shape
    assert S == 1 and b_t2.shape == (2 * Rp, Cc) and b_t2.is_contiguous() and T.shape == (M, Rp) and T.is_contiguous()
    assert dh.dtype == BF16 and dh.is_contiguous() and dsc.dtype == F32 and dsc.numel() == Rp and dsc.is_contiguous()
    dx_out = torch.empty_like(x)
    g_out = torch.empty((M, Cc), device=x.device, dtype=BF16)
    dT = torch.empty((M, 3 * Rp), device=x.device, dtype=BF16)
    L.check(L.lib().cara_ln_bwd_rows(dh.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
                                     _p(dx_in), dx_out.data_ptr(), g_out.data_ptr(), _p(rowscale), rows_per_sample, M, Cc,
                                     b_t2.data_ptr(), scales.data_ptr(), Rp, T.data_ptr(), dT.data_ptr(), dsc.data_ptr(),
                                     st), "cara_ln_bwd_rows")
    return dx_out, g_out, dT


def factor_operands(F, Rp):
    """fp32 factor [..., rows, R] -> (ext bf16 [..., rows, 3Rp] = [hi|hi|lo], t2 bf16 [..., 2Rp, rows] = [hi^T; lo^T])."""
    F = F.detach().float().contiguous()
    st = _prep(F)
    rows, R = F.shape[-2], F.shape[-1]
    lead = tuple(F.shape[:-2])
    batch = 1
    for d in lead:
        batch *= d
    ext = torch.empty(lead + (rows, 3 * Rp), device=F.device, dtype=BF16)
    t2 = torch.empty(lead + (2 * Rp, rows), device=F.device, dtype=BF16)
    L.check(L.lib().cara_factor_operands(F.data_ptr(), ext.data_ptr(), t2.data_ptr(), batch, rows, R, Rp, st),
            "cara_factor_operands")
    return ext, t2


def stage_terms(desc_fill, backward, anchor):
    """One launch of the CP-factor staging (backward = 0) or of its chain rule (1); ``desc_fill`` maps field names of
    ``cara_stage_desc`` to ints / tensors (None = NULL).  ``anchor`` is any CUDA tensor of the call (device, stream)."""
    st = _prep(anchor)
    d = L.StageDesc()
    for k, v in desc_fill.items():
        if v is None:
            continue
        if isinstance(v, torch.Tensor):
            if not v.is_cuda:
                raise L.CaraLibraryError("cara_stage_terms needs CUDA tensors (no CPU fallback)")
            setattr(d, k, v.data_ptr())
        else:
            setattr(d, k, int(v))
    L.check(L.lib().cara_stage_terms(C.byref(d), int(backward), st), "cara_stage_terms")


def adapter_rows_fwd(x, a_t2, scales):
    """x bf16 [M,K]; a_t2 bf16 [2Rp,K]; scales fp32 [S,Rp] -> (T fp32 [M,Rp], Uhat bf16 [M,S*3Rp])."""
    st = _prep(x)
    M, K = x.shape
    S, Rp = scales.shape
    assert a_t2.shape == (2 * Rp, K) and a_t2.is_contiguous() and scales.is_contiguous() and x.stride(1) == 1
    T = torch.empty((M, Rp), device=x.device, dtype=F32)
    U = torch.empty((M, S * 3 * Rp), device=x.device, dtype=BF16)
    L.check(L.lib().cara_adapter_rows_fwd(x.data_ptr(), x.stride(0), M, K, a_t2.data_ptr(), scales.data_ptr(), S, Rp,
                                          T.data_ptr(), U.data_ptr(), st), "cara_adapter_rows_fwd")
    return T, U


def adapter_rows_bwd(g, b_t2, scales, T, dsc=None):
    """g bf16 [M,N]; b_t2 bf16 [2Rp,N/S]; scales [S,Rp]; T fp32 [M,Rp] -> (dThat bf16 [M,3Rp], dscales fp32 [S,Rp]).
    ``dsc`` (optional) is a pre-zeroed fp32 [S,Rp] buffer to accumulate into."""
    st = _prep(g)
    M, N = g.shape
    S, Rp = scales.shape
    assert b_t2.shape == (2 * Rp, N // S) and b_t2.is_contiguous() and T.shape == (M, Rp) and g.stride(1) == 1
    dT = torch.empty((M, 3 * Rp), device=g.device, dtype=BF16)
    if dsc is None:
        dsc = torch.zeros((S, Rp), device=g.device, dtype=F32)
    L.check(L.lib().cara_adapter_rows_bwd(g.data_ptr(), g.stride(0), M, N, S, b_t2.data_ptr(), scales.data_ptr(), Rp,
                                          T.data_ptr(), dT.data_ptr(), dsc.data_ptr(), st), "cara_adapter_rows_bwd")
    return dT, dsc


def adapter_cols(x, v, slices, Rp, want_colsum=False, out=None, cs=None):
    """out [Kc/slices, Rp] = sum_s x[:, slice s]^T (vhi + vlo)[:, slice s]; v bf16 [M, slices*3Rp];
    colsum [Kc] = column sums of x.  ``out`` / ``cs`` (optional) are pre-zeroed buffers to accumulate into."""
    st = _prep(x)
    M, Kc = x.shape
    assert v.shape == (M, slices * 3 * Rp) and x.stride(1) == 1 and v.stride(1) == 1
    if out is None:
        out = torch.zeros((Kc // slices, Rp), device=x.device, dtype=F32)
    if cs is None and want_colsum:
        cs = torch.zeros(Kc, device=x.device, dtype=F32)
    L.check(L.lib().cara_adapter_cols(x.data_ptr(), x.stride(0), M, Kc, v.data_ptr(), v.stride(0), slices, Rp,
                                      out.data_ptr(), _p(cs), st), "cara_adapter_cols")
    return out, cs


def attn_fwd(qkv, B, N, H, D, scale, train=True):
    """-> (o bf16 [B*N, H*D], o_lo, lse); o_lo / lse are None when train is False."""
    st = _prep(qkv)
    assert qkv.dtype == BF16 and qkv.is_contiguous() and qkv.numel() == B * N * 3 * H * D
    o = torch.empty((B * N, H * D), device=qkv.device, dtype=BF16)
    o_lo = torch.empty_like(o) if train else None
    lse = torch.empty((B, H, N), device=qkv.device, dtype=F32) if train else None
    L.check(L.lib().cara_attn_fwd(qkv.data_ptr(), o.data_ptr(), _p(o_lo), _p(lse), B, N, H, D, scale, st),
            "cara_attn_fwd")
    return o, o_lo, lse


def attn_delta_fusable(N, D):
    """Shapes whose softmax-backward row term the output projection's dX GEMM can emit (EPI_DELTA): the tcgen05
    attention path (any N), head dim = one 64-column epilogue step."""
    return delta_in_gemm and D == 64 and (int(os.environ.get("CARA_ATTN_TC", "3")) & 2) != 0


def attn_bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, scale, delta=None):
    """``delta`` [B,H,N] fp32: already computed (cara_gemm_cp, EPI_DELTA) -- the pre-pass over dO and O is skipped."""
    st = _prep(qkv)
    assert d_o.is_contiguous() and d_o.dtype == BF16
    dqkv = torch.empty_like(qkv)
    pre = delta is not None
    if not pre:
        delta = torch.empty((B, H, N), device=qkv.device, dtype=F32)
    L.check(L.lib().cara_attn_bwd(qkv.data_ptr(), None if pre else o.data_ptr(), None if pre else o_lo.data_ptr(),
                                  lse.data_ptr(), d_o.data_ptr(), dqkv.data_ptr(), delta.data_ptr(), B, N, H, D, scale, st),
            "cara_attn_bwd")
    return dqkv


# The largest N the whole-head D = 80 kernels (cara_attn_fwd / cara_attn_bwd) take: the head's tiles must fit in shared
# memory.  Above them ops.AttnCoreFunction runs the key-tiled kernels (cara_attn_tiled_fwd / _bwd), which take any N.
D80_WHOLE_HEAD_MAX_N = {"fwd": 432, "bwd": 320}


def attn_tiled_fwd(qkv, B, N, H, D, scale, train=True):
    """``attn_fwd`` on the key-tiled D = 80 kernels (any N): -> (o, o_lo, lse); o_lo / lse are None when train is False."""
    st = _prep(qkv)
    assert qkv.dtype == BF16 and qkv.is_contiguous() and qkv.numel() == B * N * 3 * H * D
    o = torch.empty((B * N, H * D), device=qkv.device, dtype=BF16)
    o_lo = torch.empty_like(o) if train else None
    lse = torch.empty((B, H, N), device=qkv.device, dtype=F32) if train else None
    L.check(L.lib().cara_attn_tiled_fwd(qkv.data_ptr(), o.data_ptr(), _p(o_lo), _p(lse), B, N, H, D, scale, st),
            "cara_attn_tiled_fwd")
    return o, o_lo, lse


def attn_tiled_bwd(qkv, o, o_lo, lse, d_o, B, N, H, D, scale):
    """``attn_bwd`` on the key-tiled D = 80 kernels (any N); always runs its own delta pre-pass (o and o_lo needed)."""
    st = _prep(qkv)
    assert d_o.is_contiguous() and d_o.dtype == BF16
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((B, H, N), device=qkv.device, dtype=F32)
    L.check(L.lib().cara_attn_tiled_bwd(qkv.data_ptr(), _p(o), _p(o_lo), lse.data_ptr(), d_o.data_ptr(), dqkv.data_ptr(),
                                        delta.data_ptr(), B, N, H, D, scale, st), "cara_attn_tiled_bwd")
    return dqkv


def gelu_f32(x, dy=None):
    """fp32 mode: GELU(x) (dy None) or dy * GELU'(x), exact erf."""
    st = _prep(x)
    assert x.dtype == F32 and x.is_contiguous() and (dy is None or (dy.dtype == F32 and dy.is_contiguous()))
    out = torch.empty_like(x)
    L.check(L.lib().cara_gelu_f32(_p(dy), x.data_ptr(), out.data_ptr(), x.numel(), st), "cara_gelu_f32")
    return out


def attn_f32_fwd(qkv, B, N, H, D, scale, train=True):
    """fp32 mode attention core: qkv fp32 [B,N,3,H,D] -> (o fp32 [B*N, H*D], lse [B,H,N] or None)."""
    st = _prep(qkv)
    assert qkv.dtype == F32 and qkv.is_contiguous() and qkv.numel() == B * N * 3 * H * D
    o = torch.empty((B * N, H * D), device=qkv.device, dtype=F32)
    lse = torch.empty((B, H, N), device=qkv.device, dtype=F32) if train else None
    L.check(L.lib().cara_attn_f32(qkv.data_ptr(), o.data_ptr(), _p(lse), None, None, B, N, H, D, scale, st), "cara_attn_f32")
    return o, lse


def attn_f32_bwd(qkv, o, lse, d_o, B, N, H, D, scale):
    st = _prep(qkv)
    assert d_o.dtype == F32 and d_o.is_contiguous()
    dqkv = torch.empty_like(qkv)
    L.check(L.lib().cara_attn_f32(qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), d_o.data_ptr(), dqkv.data_ptr(), B, N, H, D,
                                  scale, st), "cara_attn_f32")
    return dqkv


def patchify(img, P, Kp):
    st = _prep(img)
    B, Cin, S, _ = img.shape
    assert img.dtype == F32 and img.is_contiguous()
    out = torch.empty((B * (S // P) ** 2, Kp), device=img.device, dtype=BF16)
    L.check(L.lib().cara_patchify(img.data_ptr(), out.data_ptr(), B, Cin, S, P, Kp, st), "cara_patchify")
    return out


def assemble_tokens(pe, cls, pos, B, N, Cc):
    st = _prep(pe)
    x = torch.empty((B * N, Cc), device=pe.device, dtype=F32)
    L.check(L.lib().cara_assemble_tokens(pe.data_ptr(), cls.data_ptr(), pos.data_ptr(), x.data_ptr(), B, N, Cc, st),
            "cara_assemble_tokens")
    return x


_MERGE_RANKS = (4, 8, 16, 32, 64)


def merge_weights(W, A, Bf, cs, out=None):
    """W fp32 [N,K], A fp32 [K,R], Bf fp32 [N/S,R], cs fp32 [S,R] -> bf16 [N,K] = W + sum_r (Bf (.) cs) A^T.
    Any rank up to 64: the factors are zero-padded to the next rank the kernel is instantiated for."""
    st = _prep(W)
    N, K = W.shape
    S, R = cs.shape
    Rk = next((r for r in _MERGE_RANKS if r >= R), None)
    if Rk is None:
        raise L.CaraLibraryError("cara_merge_weights: rank %d > %d is not supported" % (R, _MERGE_RANKS[-1]))
    if Rk != R:
        pad = lambda t: torch.nn.functional.pad(t, (0, Rk - R))                       # noqa: E731
        A, Bf, cs = pad(A), pad(Bf), pad(cs)
    A, Bf, cs = A.contiguous(), Bf.contiguous(), cs.contiguous()
    assert W.dtype == F32 and W.is_contiguous() and A.dtype == F32 and Bf.dtype == F32 and cs.dtype == F32
    if out is None:
        out = torch.empty((N, K), device=W.device, dtype=BF16)
    L.check(L.lib().cara_merge_weights(W.data_ptr(), A.data_ptr(), Bf.data_ptr(), cs.data_ptr(), out.data_ptr(),
                                       N, K, S, Rk, st), "cara_merge_weights")
    return out


def adamw_step(p, g, m, v, lr, step, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, gscale=1.0):
    global param_generation
    param_generation += 1
    st = _prep(p)
    assert p.dtype == F32 and p.is_contiguous() and g.is_contiguous()
    L.check(L.lib().cara_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, betas[0],
                                    betas[1], eps, weight_decay, step, gscale, st), "cara_adamw_step")


def adamw_step_dev(p, g, m, v, state, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, gscale=1.0):
    """AdamW with lr / step count read from the device tensor ``state`` (fp32[4], see cara_adamw_step_dev): the launch
    is graph-capturable."""
    global param_generation
    param_generation += 1
    st = _prep(p)
    assert p.dtype == F32 and p.is_contiguous() and g.is_contiguous() and state.dtype == F32 and state.numel() >= 4
    L.check(L.lib().cara_adamw_step_dev(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(),
                                        state.data_ptr(), betas[0], betas[1], eps, weight_decay, gscale, st),
            "cara_adamw_step_dev")


_SGEMM_WS_FLOATS = 1 << 22          # 16 MB of split-K partial sums per device (stream-ordered reuse)
_sgemm_ws = {}


def _sgemm_workspace(device):
    ws = _sgemm_ws.get(device)
    if ws is None:
        ws = _sgemm_ws[device] = torch.empty(_SGEMM_WS_FLOATS, device=device, dtype=F32)
    return ws


def sgemm(A, B, bias=None, out=None, alpha=1.0, beta=0.0):
    """fp32 C = alpha * A @ B + beta * C + bias for arbitrary-stride 2-D views."""
    st = _prep(A)
    M, K = A.shape
    N = B.shape[1]
    assert A.dtype == F32 and B.dtype == F32 and B.shape[0] == K
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=F32)
    ws = _sgemm_workspace(A.device) if M * N <= _SGEMM_WS_FLOATS // 4 else None   # small outputs only (split-K)
    L.check(L.lib().cara_sgemm(A.data_ptr(), A.stride(0), A.stride(1), B.data_ptr(), B.stride(0), B.stride(1),
                               out.data_ptr(), out.stride(0), _p(bias), M, N, K, alpha, beta, _p(ws),
                               0 if ws is None else ws.numel(), st), "cara_sgemm")
    return out

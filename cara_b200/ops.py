"""Autograd glue over the C-ABI kernels: each class is one differentiable unit of the CaRA hot path.

Forward/backward math follows SURVEY Appendix A.1/A.2 (verified there against the reference's autograd):
for every adapted projection  Y = X W^T + b_eff + sum_slices [(X A) (.) cs_s] B^T  and, with G = dY,
  dX = G W + dThat A^T,  dThat = sum_s cs_s (.) (G_s B),  dA = X^T dThat,  dB = sum_s G_s^T Uhat_s,
  dcs_s = sum_m (G_s B) (.) (X A),  db_eff = sum_m G.
Frozen weights receive no gradient (vit_cp.py:176-182) and no [K,N]-sized dW is ever formed.
"""
import torch

from . import _lib as L
from . import kernels as K

BF16, F32 = torch.bfloat16, torch.float32
SIDE_RPS = (16, 32)   # padded ranks the projection GEMM's side tiles cover (CARA_SIDE_TILES=1)


class FrozenLinear:
    """bf16 working copies of one frozen nn.Linear: W [N,K] for the forward GEMM, W^T [K,N] for dX."""

    __slots__ = ("w", "wt", "bias", "key")

    def __init__(self, lin):
        self.refresh(lin)

    def refresh(self, lin):
        w = lin.weight.detach()
        self.w = w.to(BF16).contiguous()
        self.wt = w.t().to(BF16).contiguous()
        self.bias = None if lin.bias is None else lin.bias.detach().to(F32).contiguous()
        self.key = FrozenLinear.key_of(lin)

    @staticmethod
    def key_of(lin):
        return (lin.weight.data_ptr(), lin.weight._version, lin.weight.device,
                None if lin.bias is None else (lin.bias.data_ptr(), lin.bias._version))

    @staticmethod
    def of(lin):
        fz = lin.__dict__.get("_cara_frozen")
        key = FrozenLinear.key_of(lin)
        if fz is None or fz.key != key:
            fz = FrozenLinear(lin)
            lin.__dict__["_cara_frozen"] = fz
        return fz


class AdapterOperands:
    """bf16 (hi, lo) forms of one projection's staged factors (not differentiable; built once per step).
    ``a_ext``/``b_ext``: [rows, 3Rp] = [hi|hi|lo] (adapter segment of the GEMM); ``a_t2``/``b_t2``: [2Rp, rows]
    (skinny kernels); ``cs_pad``: fp32 [slices, Rp]."""

    __slots__ = ("a_t2", "a_ext", "b_t2", "b_ext", "cs_pad", "rank", "rp", "slices")

    def __init__(self, a_ext, a_t2, b_ext, b_t2, cs_pad, rank):
        self.a_ext, self.a_t2, self.b_ext, self.b_t2, self.cs_pad = a_ext, a_t2, b_ext, b_t2, cs_pad
        self.rank, self.rp, self.slices = rank, cs_pad.shape[1], cs_pad.shape[0]

    @staticmethod
    def build(A, Bf, cs):
        R = A.shape[1]
        Rp = K.round_rank(R)
        a_ext, a_t2 = K.factor_operands(A, Rp)
        b_ext, b_t2 = K.factor_operands(Bf, Rp)
        cs_pad = torch.nn.functional.pad(cs.detach().to(F32), (0, Rp - R)).contiguous()
        return AdapterOperands(a_ext, a_t2, b_ext, b_t2, cs_pad, R)


class GradSink:
    """One zero-filled fp32 buffer per root forward that every projection's backward kernels accumulate their
    factor gradients into (the kernels add atomically anyway).  Without it each of the 4L projections hands
    autograd four fresh tensors, and the engine spends ~350 tiny fill / add launches per step summing them into
    the shared ``CP_*`` terms.  Per projection kind k (0 qkv, 1 proj, 2 fc1, 3 fc2):
    ``dA[k]`` [K,Rp] (fc2: [L,4C,Rp], its in-side factor is per layer), ``dB[k]`` [N/S,Rp], ``dcs[k]`` [L,S,Rp],
    ``dbias[k]`` [L,N] (None for qkv).  The gradients are returned to autograd once per kind, by the last
    backward of that kind (``release``); the others return None."""

    def __init__(self, L_, C, Rp, device):
        shapes = {"dA0": (C, Rp), "dB0": (C, Rp), "dcs0": (L_, 3, Rp),
                  "dA1": (C, Rp), "dB1": (C, Rp), "dcs1": (L_, 1, Rp), "db1": (L_, C),
                  "dA2": (C, Rp), "dB2": (C, Rp), "dcs2": (L_, 4, Rp), "db2": (L_, 4 * C),
                  "dA3": (L_, 4 * C, Rp), "dB3": (C, Rp), "dcs3": (L_, 1, Rp), "db3": (L_, C)}
        sizes = [int(torch.Size(v).numel()) for v in shapes.values()]
        self.buf = torch.zeros(sum(sizes), device=device, dtype=F32)
        self.t = {k: v.view(shapes[k]) for k, v in zip(shapes, torch.split(self.buf, sizes))}
        self.pending = [0, 0, 0, 0]

    def views(self, kind, layer, need_bias):
        dA = self.t["dA%d" % kind]
        if kind == 3:
            dA = dA[layer]
        db = self.t["db%d" % kind][layer] if (need_bias and kind > 0) else None
        return dA, self.t["dcs%d" % kind][layer], self.t["dB%d" % kind], db

    def release(self, kind, R, need_bias):
        """-> (dA, dcs, dB, dbias) for autograd if this was the last pending backward of ``kind``, else Nones."""
        self.pending[kind] -= 1
        if self.pending[kind] > 0:
            return None, None, None, None
        db = self.t["db%d" % kind] if (need_bias and kind > 0) else None
        return self.t["dA%d" % kind][..., :R], self.t["dcs%d" % kind][..., :R], self.t["dB%d" % kind][..., :R], db


class RowsLink:
    """Hand-over between a LayerNorm kernel and the adapted projection next to it (csrc/ln_rows.cu).
    Forward link (LayerNorm -> the qkv / fc1 it feeds): ``ops`` = that projection's operands, set by the caller; the
    LayerNorm deposits ``T`` / ``U`` and the projection skips its rows pass.
    Backward link (proj / fc2 -> the LayerNorm that adds its output to the residual stream): the projection's forward
    deposits ``ops``, its saved ``T`` and the ``dcs`` accumulator; the LayerNorm's backward -- whose g_out IS that
    projection's incoming gradient -- deposits ``dT`` and the projection's backward skips its rows pass."""

    __slots__ = ("ops", "want_T", "T", "U", "dT", "dcs")

    def __init__(self, ops=None, want_T=True):
        self.ops, self.want_T = ops, want_T        # want_T: keep T for a backward (autograd is off inside Function.forward)
        self.T = self.U = self.dT = self.dcs = None


def _cp_linear_fwd(x, fz, bias_eff, ops, epi=L.EPI_NONE, want_pre=True, train=True, pre=None):
    """The frozen product + the adapter segment (cara.py:35,57,81,92 without the delta weight).  The rank-R row
    contraction T = x A, Uhat_s = cs_s (.) T that feeds the segment comes from the LayerNorm kernel that produced x
    (``pre``, a filled forward RowsLink), or runs as its own pass (default) or, with CARA_SIDE_TILES=1, as side tiles
    of the same GEMM launch (Rp = 16 / 32; an Rp = 64 projection keeps its own pass)."""
    T = U = None
    if ops is not None and pre is not None and pre.U is not None:
        T, U = pre.T, pre.U
        y = K.gemm_cp(x, fz.w, bias=bias_eff, a1=U, b1=ops.b_ext, ext_slices=ops.slices, epi=epi, want_pre=want_pre)
    elif ops is not None and not (K.side_tiles and epi == L.EPI_NONE and ops.rp in SIDE_RPS):
        # default: the row contraction T = x A, Uhat_s = cs_s (.) T as its own HBM-bound pass, then the GEMM
        T, U = K.adapter_rows_fwd(x, ops.a_t2, ops.cs_pad)
        y = K.gemm_cp(x, fz.w, bias=bias_eff, a1=U, b1=ops.b_ext, ext_slices=ops.slices, epi=epi, want_pre=want_pre)
    elif ops is not None:
        M = x.shape[0]
        T = torch.empty((M, ops.rp), device=x.device, dtype=F32) if train else None
        U = torch.empty((M, ops.slices * 3 * ops.rp), device=x.device, dtype=BF16)
        side = K.Side(L.SIDE_FWD, ops.a_t2, ops.cs_pad, T, U)
        y = K.gemm_cp(x, fz.w, bias=bias_eff, a1=U, b1=ops.b_ext, ext_slices=ops.slices, epi=epi, want_pre=want_pre,
                      side=side)
    else:
        y = K.gemm_cp(x, fz.w, bias=bias_eff, epi=epi, want_pre=want_pre)
    return y, T, U


def _cp_linear_bwd(G, x, fz, ops, T, U, need_dx, need_bias, dgelu_aux=None, sink=None, delta=None, dT_pre=None):
    """Returns (dx, dA, dcs, dB, dbias).  ``sink`` = (GradSink, kind, layer): accumulate the factor gradients
    there and hand them to autograd once per projection kind (see GradSink).  ``delta`` (output projection of the
    attention branch only) = (o, o_lo, delta_out, seq_n): the dX GEMM's epilogue also emits rowsum(dX (.) O)."""
    epi = L.EPI_DGELU if dgelu_aux is not None else (L.EPI_DELTA if delta is not None else L.EPI_NONE)
    if ops is None:
        dx = K.gemm_cp(G, fz.wt, epi=epi, aux=dgelu_aux, delta=delta) if need_dx else None
        return dx, None, None, None, None
    R, Rp, S = ops.rank, ops.rp, ops.slices
    Kin, N = x.shape[1], G.shape[1]
    w = N // S
    if sink is not None:
        dA, dcs, dB, colsum = sink[0].views(sink[1], sink[2], need_bias)
    else:
        # one zero fill for every atomically accumulated output of this projection's backward
        sizes = (S * Rp, Kin * Rp, w * Rp, N if need_bias else 0)
        z = torch.zeros(sum(sizes), device=G.device, dtype=F32)
        zs = torch.split(z, sizes)
        dcs, dA, dB = zs[0].view(S, Rp), zs[1].view(Kin, Rp), zs[2].view(w, Rp)
        colsum = zs[3] if need_bias else None
    if dT_pre is not None or not (K.side_tiles and epi == L.EPI_NONE and Rp in SIDE_RPS):
        # the three readers of G run back to back: for the C-wide projections G (77 MB at ViT-B) stays in the 126 MB L2
        # (dT_pre: dThat and dcs already came out of the LayerNorm backward that produced G)
        dT = dT_pre if dT_pre is not None else K.adapter_rows_bwd(G, ops.b_t2, ops.cs_pad, T, dsc=dcs)[0]
        K.adapter_cols(G, U, S, Rp, want_colsum=need_bias, out=dB, cs=colsum)
        dx = K.gemm_cp(G, fz.wt, a1=dT, b1=ops.a_ext, ext_slices=1, epi=epi, aux=dgelu_aux, delta=delta) if need_dx else None
        K.adapter_cols(x, dT, 1, Rp, out=dA)
        if sink is not None:
            return (dx,) + sink[0].release(sink[1], R, need_bias)
        return dx, dA[:, :R], dcs[:, :R], dB[:, :R], colsum
    K.adapter_cols(G, U, S, Rp, want_colsum=need_bias, out=dB, cs=colsum)
    dx = None
    if need_dx:
        # dX GEMM; its side tiles contract the same G panels with B: dThat = sum_s cs_s (.) (G_s B), dcs += dU (.) T
        dT = torch.empty((G.shape[0], 3 * Rp), device=G.device, dtype=BF16)
        side = K.Side(L.SIDE_BWD, ops.b_t2, ops.cs_pad, T, dT, dcs)
        dx = K.gemm_cp(G, fz.wt, a1=dT, b1=ops.a_ext, ext_slices=1, epi=epi, aux=dgelu_aux, side=side)
    else:
        dT, _ = K.adapter_rows_bwd(G, ops.b_t2, ops.cs_pad, T, dsc=dcs)      # the side tiles alone (first block's qkv)
    K.adapter_cols(x, dT, 1, Rp, out=dA)
    if sink is not None:
        return (dx,) + sink[0].release(sink[1], R, need_bias)
    return dx, dA[:, :R], dcs[:, :R], dB[:, :R], colsum


def _arm_backward_link(post, ops, T, sink, train):
    """Forward of proj / fc2: let the LayerNorm backward that will produce this projection's incoming gradient also
    run its dU = G B contraction (needs the gradient sink: dcs is accumulated in place)."""
    if post is not None and train and ops is not None and sink is not None and T is not None and ops.slices == 1:
        post.ops, post.T = ops, T
        post.dcs = sink[0].t["dcs%d" % sink[1]][sink[2]]


def _take_dT(post):
    if post is None:
        return None
    dT, post.dT, post.T, post.ops, post.dcs = post.dT, None, None, None, None
    return dT


class CPLinearFunction(torch.autograd.Function):
    """One CP-adapted frozen projection (qkv: cara.py:25-42, proj: cara.py:50-58)."""

    @staticmethod
    def forward(ctx, x, A, cs, Bf, bias_eff, fz, ops, sink=None, link=None, pre=None, post=None):
        """Without ``sink``: A [K,R], cs [S,R], Bf [N/S,R], bias_eff [N] are this layer's terms.  With ``sink`` =
        (GradSink, kind, layer): cs [L,S,R] and bias_eff [L,N] (and A [L,4C,R] for fc2) are the stacked terms of
        all layers -- autograd sees one gradient per kind instead of one per layer.  ``link`` (an ``AttnLink``, output
        projection only): x is the attention core's output and this backward's dX GEMM also writes the core's
        softmax-backward row term (EPI_DELTA)."""
        bias = bias_eff if (bias_eff is None or sink is None) else bias_eff[sink[2]]
        train = any(ctx.needs_input_grad)
        y, T, U = _cp_linear_fwd(x, fz, bias if bias is not None else fz.bias, ops, train=train, pre=pre)
        if sink is not None and train:
            sink[0].pending[sink[1]] += 1
        _arm_backward_link(post, ops, T, sink, train)
        ctx.fz, ctx.ops, ctx.sink, ctx.link, ctx.post = fz, ops, sink, link, post
        ctx.save_for_backward(x, T, U)
        return y

    @staticmethod
    def backward(ctx, G):
        x, T, U = ctx.saved_tensors
        ni = ctx.needs_input_grad
        link, delta = ctx.link, None
        if link is not None and link.o_lo is not None and ni[0]:
            link.delta = torch.empty(link.shape, device=G.device, dtype=F32)
            delta = (x, link.o_lo, link.delta, link.shape[2])
        dx, dA, dcs, dB, dbias = _cp_linear_bwd(G.contiguous(), x, ctx.fz, ctx.ops, T, U, ni[0], ni[4], sink=ctx.sink,
                                                delta=delta, dT_pre=_take_dT(ctx.post))
        return dx, dA, dcs, dB, dbias, None, None, None, None, None, None


class CPMlpFunction(torch.autograd.Function):
    """cp_mlp (cara.py:72-95): fc1 + adapter -> exact-erf GELU -> fc2 + adapter, as one unit so the
    GELU and its derivative are both evaluated in the fc1 GEMM epilogue (the derivative is what is kept for backward:
    the fc2 dX GEMM epilogue only multiplies by it)."""

    @staticmethod
    def forward(ctx, x, A1, cs1, B1, bias1, A2, cs2, B2, bias2, fz1, ops1, fz2, ops2, sink1=None, sink2=None,
                pre=None, post=None):
        train = any(ctx.needs_input_grad)
        if sink1 is not None:                 # stacked terms of all layers (see CPLinearFunction.forward)
            bias1 = None if bias1 is None else bias1[sink1[2]]
            bias2 = None if bias2 is None else bias2[sink2[2]]
            if train:
                sink1[0].pending[sink1[1]] += 1
                sink2[0].pending[sink2[1]] += 1
        # gp = gelu'(u), g = GELU(u) from the fc1 epilogue (u = fc1 pre-activation, never stored)
        (gp, g), T1, U1 = _cp_linear_fwd(x, fz1, bias1 if bias1 is not None else fz1.bias, ops1, epi=L.EPI_GELU,
                                         want_pre=train, train=train, pre=pre)
        y, T2, U2 = _cp_linear_fwd(g, fz2, bias2 if bias2 is not None else fz2.bias, ops2, train=train)
        _arm_backward_link(post, ops2, T2, sink2, train)
        ctx.post = post
        ctx.fz1, ctx.ops1, ctx.fz2, ctx.ops2 = fz1, ops1, fz2, ops2
        ctx.sink1, ctx.sink2 = sink1, sink2
        ctx.save_for_backward(x, gp, g, T1, U1, T2, U2)
        return y

    @staticmethod
    def backward(ctx, G):
        x, gp, g, T1, U1, T2, U2 = ctx.saved_tensors
        ni = ctx.needs_input_grad
        du, dA2, dcs2, dB2, db2 = _cp_linear_bwd(G.contiguous(), g, ctx.fz2, ctx.ops2, T2, U2, True, ni[8],
                                                 dgelu_aux=gp, sink=ctx.sink2, dT_pre=_take_dT(ctx.post))
        dx, dA1, dcs1, dB1, db1 = _cp_linear_bwd(du, x, ctx.fz1, ctx.ops1, T1, U1, ni[0], ni[4], sink=ctx.sink1)
        return dx, dA1, dcs1, dB1, db1, dA2, dcs2, dB2, db2, None, None, None, None, None, None, None, None


class AttnLink:
    """Hand-over between the attention core and the output projection that consumes it: the projection's dX GEMM
    holds every dO tile in registers, so its epilogue (EPI_DELTA) writes rowsum(dO (.) O) for the core's backward and
    the separate 232 MB pass over dO and O goes away.  Forward: the core deposits o_lo and the [B,H,N] shape;
    backward: the projection deposits ``delta``, the core takes it."""

    __slots__ = ("o_lo", "shape", "delta")

    def __init__(self):
        self.o_lo = self.shape = self.delta = None


def _d80_tiled(D, N, direction):
    """D = 80 above the whole-head kernels' shared-memory limit runs on the key-tiled kernels (any N).  Below it the
    whole-head kernels keep running, so ViT-H/14 at 224 px launches what it always did; between the two limits
    (320 < N <= 432) a whole-head forward feeds a tiled backward."""
    return D == 80 and N > K.D80_WHOLE_HEAD_MAX_N[direction]


class AttnCoreFunction(torch.autograd.Function):
    """softmax(q k^T D^-1/2) v on the fused projection's [B,N,3,H,D] output (cara.py:44-48)."""

    @staticmethod
    def forward(ctx, qkv, B, N, H, D, scale, link=None):
        fwd = K.attn_tiled_fwd if _d80_tiled(D, N, "fwd") else K.attn_fwd
        o, o_lo, lse = fwd(qkv, B, N, H, D, scale, train=ctx.needs_input_grad[0])
        ctx.dims = (B, N, H, D, scale)
        ctx.link = link
        if link is not None and o_lo is not None:
            link.o_lo, link.shape = o_lo, (B, H, N)
        ctx.save_for_backward(qkv, o, o_lo, lse)
        return o

    @staticmethod
    def backward(ctx, d_o):
        qkv, o, o_lo, lse = ctx.saved_tensors
        B, N, H, D, scale = ctx.dims
        delta = None
        if ctx.link is not None:
            delta, ctx.link.delta = ctx.link.delta, None
        if _d80_tiled(D, N, "bwd"):                        # no EPI_DELTA at D = 80: delta is None here
            return (K.attn_tiled_bwd(qkv, o, o_lo, lse, d_o.contiguous(), B, N, H, D, scale),
                    None, None, None, None, None, None)
        return (K.attn_bwd(qkv, o, o_lo, lse, d_o.contiguous(), B, N, H, D, scale, delta=delta),
                None, None, None, None, None, None)


class LayerNormFunction(torch.autograd.Function):
    """h = LN(x) for the first block / final norm (frozen affine).  x fp32 [M,C]."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, act_dtype, fl=None):
        """``fl``: forward RowsLink of the projection that consumes h (its row contraction runs in this kernel)."""
        if fl is not None and act_dtype == BF16:
            _, h, mean, rstd, fl.T, fl.U = K.ln_fwd_rows(x, gamma, beta, fl.ops.a_t2, fl.ops.cs_pad, eps=eps,
                                                         want_T=fl.want_T)
        else:
            _, h, mean, rstd = K.ln_fwd(x, gamma, beta, eps=eps, act_dtype=act_dtype)
        ctx.save_for_backward(x, mean, rstd, gamma)
        return h

    @staticmethod
    def backward(ctx, dh):
        x, mean, rstd, gamma = ctx.saved_tensors
        dx, _ = K.ln_bwd(dh.contiguous(), x, mean, rstd, gamma)
        return dx, None, None, None, None, None


class AddLayerNormFunction(torch.autograd.Function):
    """x_new = x + rowscale * delta (residual + DropPath), h = LN(x_new): timm Block's
    ``x + drop_path(f(norm(x)))`` re-associated so the add rides in the next LayerNorm's pass."""

    @staticmethod
    def forward(ctx, x, delta, rowscale, gamma, beta, eps, rows_per_sample, fl=None, bl=None):
        """``fl``: forward RowsLink of the projection that consumes h; ``bl``: backward RowsLink armed by the
        projection that produced ``delta`` (this backward's g is its incoming gradient)."""
        if fl is not None and delta.dtype == BF16:
            x_new, h, mean, rstd, fl.T, fl.U = K.ln_fwd_rows(x, gamma, beta, fl.ops.a_t2, fl.ops.cs_pad, delta=delta,
                                                             rowscale=rowscale, rows_per_sample=rows_per_sample, eps=eps,
                                                             want_T=fl.want_T)
        else:
            x_new, h, mean, rstd = K.ln_fwd(x, gamma, beta, delta=delta, rowscale=rowscale,
                                            rows_per_sample=rows_per_sample, eps=eps, act_dtype=delta.dtype)
        ctx.rps, ctx.bl = rows_per_sample, bl
        ctx.save_for_backward(x_new, mean, rstd, gamma, rowscale)
        return x_new, h

    @staticmethod
    def backward(ctx, dx_new, dh):
        x_new, mean, rstd, gamma, rowscale = ctx.saved_tensors
        if dh is None:
            dh = torch.zeros(x_new.shape, device=x_new.device, dtype=BF16)
        bl = ctx.bl
        dx_in = None if dx_new is None else dx_new.contiguous()
        if bl is not None and bl.T is not None and dh.dtype == BF16:
            dx, g, bl.dT = K.ln_bwd_rows(dh.contiguous(), x_new, mean, rstd, gamma, bl.ops.b_t2, bl.ops.cs_pad, bl.T, bl.dcs,
                                         dx_in=dx_in, rowscale=rowscale, rows_per_sample=ctx.rps)
        else:
            dx, g = K.ln_bwd(dh.contiguous(), x_new, mean, rstd, gamma, dx_in=dx_in, rowscale=rowscale,
                             rows_per_sample=ctx.rps, want_g=True)
        return dx, g, None, None, None, None, None, None, None


class HeadFunction(torch.autograd.Function):
    """logits = h W^T + b for the trainable classifier (vit_cp.py:166), fp32 SIMT GEMMs."""

    @staticmethod
    def forward(ctx, h, weight, bias):
        ctx.save_for_backward(h, weight)
        return K.sgemm(h, weight.t(), bias=bias)

    @staticmethod
    def backward(ctx, dl):
        h, weight = ctx.saved_tensors
        dl = dl.contiguous()
        dh = K.sgemm(dl, weight) if ctx.needs_input_grad[0] else None
        dw = K.sgemm(dl.t(), h)
        return dh, dw, dl.sum(0)

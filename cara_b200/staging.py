"""Per-step staging of the CP factors into the per-projection terms the kernels consume.

SURVEY Appendix A.1 table: every adapted projection is  Y = X W^T + b + s ((X A (.) c) B^T + beta).  Here the
twelve ``CP_*`` parameters of the root model (cara.py:112-125) are turned -- by ONE differentiable launch
(``StageFunction`` -> ``cara_stage_terms``; its backward is one more launch), batched over all layers -- into, per layer
and projection,
``A`` [K,R], ``cs = s*c`` [slices,R], ``B`` [N/slices,R] and ``bias = b + s*beta``; autograd carries the
kernels' gradients w.r.t. these terms back to the ``CP_*`` parameters (SURVEY A.2 chain rule).  The row maps
follow the reference's own indices: ``CP_A1[attn_idx : attn_idx+3]`` (cara.py:26), ``CP_P1[idx]`` (:51),
``CP_P1[idx : idx+4]`` / ``[idx+4 : idx+8]`` (:72-73).  Results are cached until a parameter changes.
"""
import torch

from . import kernels as K
from .ops import AdapterOperands, GradSink

BF16, F32 = torch.bfloat16, torch.float32
CP_NAMES = ("CP_A1", "CP_A2", "CP_A3", "CP_A4", "CP_P1", "CP_P2", "CP_P3", "CP_R1", "CP_R2",
            "CP_bias1", "CP_bias2", "CP_bias3")


class Terms:
    """One projection's terms.  ``A cs B bias`` are this layer's tensors (fp32 parity mode, un-sunk path);
    ``stacked`` = (A or A[L,..], cs [L,S,R], B, bias [L,N] or None) are the all-layer tensors the bf16 path hands to
    autograd together with ``sink`` = (ops.GradSink, kind, layer) when gradients are on."""
    __slots__ = ("A", "cs", "B", "bias", "ops", "stacked", "sink")

    def __init__(self, A, cs, B, bias, ops, stacked=None, sink=None):
        self.A, self.cs, self.B, self.bias, self.ops = A, cs, B, bias, ops
        self.stacked, self.sink = stacked, sink

    def autograd_args(self):
        """(A, cs, B, bias, sink) for ops.CPLinearFunction / CPMlpFunction."""
        if self.sink is not None:
            return self.stacked + (self.sink,)
        return self.A, self.cs, self.B, self.bias, None


_STAGED = ("kr", "cs_qkv", "cs_proj", "cs_fc1", "a_fc2", "cs_fc2", "b_proj", "b_fc1", "b_fc2")
_PARAMS = ("A1", "A3", "A4", "P1", "P2", "R1", "R2", "bias1", "bias2", "bias3")


def _rows_with_pitch(g):
    """An R-wide gradient as (tensor, row pitch): dense tensors have pitch R; the ``[..., :R]`` views into the Rp-wide
    gradient sink (ops.GradSink.release) are passed as they are with pitch Rp; anything else is made dense."""
    if g.stride(-1) != 1:
        g = g.contiguous()
    if g.is_contiguous():
        return g, g.shape[-1]
    pitch = expect = g.stride(-2)
    for i in range(g.dim() - 2, -1, -1):
        if g.stride(i) != expect:
            return g.contiguous(), g.shape[-1]
        expect *= g.shape[i]
    return g, pitch


class StageFunction(torch.autograd.Function):
    """CP_* parameters -> the nine staged tensors (one ``cara_stage_terms`` launch) and, in backward, the chain rule
    of SURVEY A.2 back to the parameters (one more launch) -- instead of ~30 + ~60 tiny torch kernels per step.
    ``const`` = dict(ai, pi, mi int32 [L]; s_a, s_m fp32 [L]; fb_proj [L,C], fb_fc1 [L,4C], fb_fc2 [L,C]; D; Rp; pads =
    the four zero-padded [.., Rp] outputs to fill)."""

    @staticmethod
    def forward(ctx, A1, A3, A4, P1, P2, R1, R2, bias1, bias2, bias3, const):
        ps = [t.detach().float().contiguous() for t in (A1, A3, A4, P1, P2, R1, R2, bias1, bias2, bias3)]
        R, C, L_ = ps[0].shape[1], ps[4].shape[0], const["ai"].shape[0]
        dev = ps[0].device
        new = lambda *shape: torch.empty(shape, device=dev, dtype=F32)                 # noqa: E731
        out = {"kr": new(C, R), "cs_qkv": new(L_, 3, R), "cs_proj": new(L_, 1, R), "cs_fc1": new(L_, 4, R),
               "a_fc2": new(L_, 4 * C, R), "cs_fc2": new(L_, 1, R), "b_proj": new(L_, C), "b_fc1": new(L_, 4 * C),
               "b_fc2": new(L_, C)}
        fill = {"R": R, "Rp": const["Rp"], "C": C, "D": const["D"], "L": L_}
        fill.update(dict(zip(_PARAMS, ps)))
        fill.update({k: const[k] for k in ("ai", "pi", "mi", "s_a", "s_m", "fb_proj", "fb_fc1", "fb_fc2")})
        fill.update(out)
        fill.update({k + "_pad": v for k, v in const["pads"].items()})
        K.stage_terms(fill, 0, ps[0])
        ctx.const, ctx.dims = const, (R, C, L_)
        ctx.save_for_backward(*ps)
        res = tuple(out[k] for k in _STAGED)
        return res

    @staticmethod
    def backward(ctx, *grads):
        ps = ctx.saved_tensors
        const = ctx.const
        R, C, L_ = ctx.dims
        dev = ps[0].device
        sizes = [ps[0].numel(), ps[1].numel(), ps[2].numel(), ps[3].numel(), ps[4].numel(), R, R, C, 4 * C, C]
        flat = torch.zeros(sum(sizes), device=dev, dtype=F32)            # one zero fill for all ten outputs
        outs = [v.view(p.shape) for v, p in zip(torch.split(flat, sizes), ps)]
        fill = {"R": R, "Rp": const["Rp"], "C": C, "D": const["D"], "L": L_}
        fill.update(dict(zip(_PARAMS, ps)))
        fill.update({k: const[k] for k in ("ai", "pi", "mi", "s_a", "s_m")})
        for name, g in zip(_STAGED, grads):
            if g is None:
                continue
            g = g if g.dtype == F32 else g.float()
            if name.startswith("b_"):
                g = g.contiguous()
            else:
                g, fill["ld_" + name] = _rows_with_pitch(g)
            fill["g_" + name] = g
        fill.update(dict(zip(("dA1", "dA3", "dA4", "dP1", "dP2", "dR1", "dR2", "dbias1", "dbias2", "dbias3"), outs)))
        K.stage_terms(fill, 1, ps[0])
        return tuple(outs) + (None,)


def _modules(model):
    from .vit import Attention, Mlp
    attn = [m for m in model.modules() if isinstance(m, Attention) and hasattr(m, "attn_idx")]
    mlp = [m for m in model.modules() if isinstance(m, Mlp) and hasattr(m, "idx")]
    return attn, mlp


def staged(model):
    """-> (dict id(attention module) -> (qkv Terms, proj Terms), dict id(mlp module) -> (fc1 Terms, fc2 Terms))."""
    P = {n: getattr(model, n) for n in CP_NAMES}
    attn, mlp = _modules(model)
    frozen = [m.proj.bias for m in attn] + [m.fc1.bias for m in mlp] + [m.fc2.bias for m in mlp]
    grad_on = torch.is_grad_enabled()
    token = model.__dict__.get("_cara_fwd_token")
    key = (tuple((p.data_ptr(), p._version) for p in P.values()), K.param_generation, grad_on,
           tuple(float(m.s) for m in attn + mlp), tuple((b.data_ptr(), b._version) for b in frozen),
           tuple(int(m.attn_idx) for m in attn), tuple(int(m.idx) for m in attn + mlp))
    cache = model.__dict__.get("_cara_stage")
    # With autograd on, the staged tensors carry a graph that one backward consumes: share them only among the
    # layers of ONE root forward (token set by VisionTransformer.forward_features); otherwise rebuild.
    if cache is not None and cache[0] == key and (not grad_on or (token is not None and cache[3] is token)):
        return cache[1], cache[2]
    dev = P["CP_A1"].device
    R = P["CP_A1"].shape[1]
    if R > K.MAX_RANK:
        raise NotImplementedError("rank > %d is not supported by the staged bf16 operands (got %d)" % (K.MAX_RANK, R))
    Rp = K.round_rank(R)
    C = P["CP_A2"].shape[0]
    f = {n: p.float() for n, p in P.items()}
    La, Lm = len(attn), len(mlp)
    # index / scale tensors: built once per (indices, scales) -- a host list -> device copy is a synchronous
    # transfer, which must not happen inside a CUDA-graph capture of the step
    ikey = (key[3], key[5], key[6], str(dev))
    icache = model.__dict__.get("_cara_stage_idx")
    if icache is None or icache[0] != ikey:
        icache = (ikey,
                  torch.tensor([int(m.attn_idx) for m in attn], device=dev, dtype=torch.int32),
                  torch.tensor([int(m.idx) for m in attn], device=dev, dtype=torch.int32),
                  torch.tensor([int(m.idx) for m in mlp], device=dev, dtype=torch.int32),
                  torch.tensor([float(m.s) for m in attn], device=dev, dtype=F32),
                  torch.tensor([float(m.s) for m in mlp], device=dev, dtype=F32))
        model.__dict__["_cara_stage_idx"] = icache
    _, ai, pi, mi, s_a, s_m = icache

    if La != Lm:
        raise NotImplementedError("CaRA staging expects one Attention and one Mlp per block")
    # the frozen biases never change during fine-tuning: stack them once per (pointer, version) set
    bkey = key[4]
    bcache = model.__dict__.get("_cara_stage_bias")
    if bcache is None or bcache[0] != bkey:
        bcache = (bkey, torch.stack([m.proj.bias.detach().float() for m in attn]).contiguous(),
                  torch.stack([m.fc1.bias.detach().float() for m in mlp]).contiguous(),
                  torch.stack([m.fc2.bias.detach().float() for m in mlp]).contiguous())
        model.__dict__["_cara_stage_bias"] = bcache
    # one launch: the nine staged tensors (SURVEY A.1 table) + the Rp-padded copies of the cs terms the kernels read
    zp = lambda *shape: torch.zeros(shape, device=dev, dtype=F32)                      # noqa: E731
    csq, csp, cs1, cs2 = zp(La, 3, Rp), zp(La, 1, Rp), zp(Lm, 4, Rp), zp(Lm, 1, Rp)
    const = {"ai": ai, "pi": pi, "mi": mi, "s_a": s_a, "s_m": s_m, "fb_proj": bcache[1], "fb_fc1": bcache[2],
             "fb_fc2": bcache[3], "D": C // P["CP_A3"].shape[0], "Rp": Rp,
             "pads": {"cs_qkv": csq, "cs_proj": csp, "cs_fc1": cs1, "cs_fc2": cs2}}
    kr_attn, cs_qkv, cs_proj, cs_fc1, a_fc2, cs_fc2, b_proj, b_fc1, b_fc2 = StageFunction.apply(
        f["CP_A1"], f["CP_A3"], f["CP_A4"], f["CP_P1"], f["CP_P2"], f["CP_R1"], f["CP_R2"], f["CP_bias1"], f["CP_bias2"],
        f["CP_bias3"], const)

    with torch.no_grad():
        a2_pad, a2_t = K.factor_operands(f["CP_A2"], Rp)
        kr_pad, kr_t = K.factor_operands(kr_attn, Rp)
        p2_pad, p2_t = K.factor_operands(f["CP_P2"], Rp)
        p3_pad, p3_t = K.factor_operands(f["CP_P3"], Rp)
        afc2_pad, afc2_t = K.factor_operands(a_fc2, Rp)

    # gradients on: every projection's backward accumulates into one zero-filled sink (ops.GradSink)
    sink = GradSink(max(La, Lm), C, Rp, dev) if (grad_on and La == Lm) else None
    sk = (lambda kind, i: (sink, kind, i)) if sink is not None else (lambda kind, i: None)
    amap, mmap = {}, {}
    for i, m in enumerate(attn):
        qkv = Terms(f["CP_A2"], cs_qkv[i], kr_attn, None, AdapterOperands(a2_pad, a2_t, kr_pad, kr_t, csq[i], R),
                    (f["CP_A2"], cs_qkv, kr_attn, None), sk(0, i))
        proj = Terms(f["CP_P3"], cs_proj[i], f["CP_P2"], b_proj[i],
                     AdapterOperands(p3_pad, p3_t, p2_pad, p2_t, csp[i], R),
                     (f["CP_P3"], cs_proj, f["CP_P2"], b_proj), sk(1, i))
        amap[id(m)] = (qkv, proj)
    for i, m in enumerate(mlp):
        fc1 = Terms(f["CP_P3"], cs_fc1[i], f["CP_P2"], b_fc1[i], AdapterOperands(p3_pad, p3_t, p2_pad, p2_t, cs1[i], R),
                    (f["CP_P3"], cs_fc1, f["CP_P2"], b_fc1), sk(2, i))
        fc2 = Terms(a_fc2[i], cs_fc2[i], f["CP_P3"], b_fc2[i],
                    AdapterOperands(afc2_pad[i], afc2_t[i], p3_pad, p3_t, cs2[i], R),
                    (a_fc2, cs_fc2, f["CP_P3"], b_fc2), sk(3, i))
        mmap[id(m)] = (fc1, fc2)
    model.__dict__["_cara_stage"] = (key, amap, mmap, token)
    return amap, mmap

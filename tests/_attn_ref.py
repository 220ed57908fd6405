"""fp64 reference of the attention core and the per-head comparison the attention kernel tests share (never imported
by the product).  The head size D is read from the tensors: [B, N, 3, H, D] for qkv."""
import math

import torch

BF16 = torch.bfloat16
BARS = {"o": 6e-3, "o+o_lo": 3e-3, "lse": 1e-4, "dq": 1.2e-2, "dk": 1.2e-2, "dv": 1.2e-2}
# N = 1: the exact dq and dk are 0 (one key, p = 1), so they are bounded absolutely, per head, by ZERO_GRAD_BAR x the
# head's |dv|.  What is left is the fp32 difference between dO . v and delta = dO . (o + o_lo) that bf16(dS) carries:
# measured on a B200 at most 1.6e-7 (D = 64) and 2.5e-7 (D = 80).
ZERO_GRAD_BAR = 1e-5


def ref_attention(qkv, d_o, scale):
    """fp64 forward and backward of softmax(q k^T scale) v, qkv [B,N,3,H,D], d_o [B*N, H*D] ->
    (o [B,N,H,D], lse [B,H,N] base 2, dqkv [B,N,3,H,D]), one sample at a time."""
    B, N, _, H, D = qkv.shape
    o, lse, dqkv = [], [], []
    for b in range(B):
        q, k, v = [t.double() for t in qkv[b].permute(1, 2, 0, 3)]               # [H,N,D]
        s = (q @ k.transpose(-1, -2)) * scale
        ls = torch.logsumexp(s, -1)
        p = torch.exp(s - ls[..., None])
        ob = p @ v
        o.append(ob.transpose(0, 1))
        lse.append(ls / math.log(2.0))
        if d_o is not None:
            do = d_o.view(B, N, H, D)[b].double().transpose(0, 1)                   # [H,N,D]
            dp = do @ v.transpose(-1, -2)
            ds = p * (dp - (do * ob).sum(-1, keepdim=True))
            dqkv.append(torch.stack([(ds @ k) * scale, (ds.transpose(-1, -2) @ q) * scale, p.transpose(-1, -2) @ do],
                                    0).permute(2, 0, 1, 3))
    return torch.stack(o), torch.stack(lse), (torch.stack(dqkv) if dqkv else None)


def head_norms(a, head_dim):
    """L2 norm per (sample, head) of a [B, N, (3,) H, D] tensor whose head axis is ``head_dim`` -> [B, H]."""
    return a.double().movedim(head_dim, 1).flatten(2).norm(dim=-1)


def worst_head(a, b, head_dim):
    """max over (sample, head) of the relative L2 error; ``head_dim`` is the index of the head axis of [B, N, (3,) H, D]
    tensors, or None for lse [B, H, N]."""
    a, b = a.double(), b.double()
    if head_dim is None:
        num = (a - b).norm(dim=-1)
        den = b.norm(dim=-1)
    else:
        num, den = head_norms(a - b, head_dim), head_norms(b, head_dim)
    return float((num / den.clamp_min(1e-30)).max())


def check(K, qkv, B, N, H, seed=1, samples=None, backward=True):
    """Run the forward (and the backward) and hold every output to BARS, per head, against the fp64 reference of the
    samples listed in ``samples`` (default: all).  The inference form must be bit-identical to the training o.
    Returns (o, lse, dqkv or None, {output: worst-head error})."""
    D = qkv.shape[-1]
    scale = D ** -0.5
    g = torch.Generator(device="cuda").manual_seed(seed)
    o, o_lo, lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale)
    d_o = dqkv = None
    if backward:
        d_o = torch.randn(B * N, H * D, device="cuda", generator=g).to(BF16)
        dqkv = K.attn_bwd(qkv.view(-1), o, o_lo, lse, d_o, B, N, H, D, scale).view(B, N, 3, H, D)
    keep = list(range(B)) if samples is None else samples
    ro, rl, rd = ref_attention(qkv[keep], None if d_o is None else d_o.view(B, N, H * D)[keep].reshape(-1, H * D), scale)
    o4, olo4 = o.view(B, N, H, D)[keep], o_lo.view(B, N, H, D)[keep]
    errs = {"o": worst_head(o4, ro, 2), "o+o_lo": worst_head(o4.double() + olo4.double(), ro, 2),
            "lse": worst_head(lse[keep], rl, None)}
    bars = dict(BARS)
    if backward:
        mine = dqkv[keep]
        for i, name in enumerate("qkv"):
            errs["d" + name] = worst_head(mine[:, :, i], rd[:, :, i], 2)
        if N == 1:
            dv = head_norms(rd[:, :, 2], 2).clamp_min(1e-30)
            for i, name in ((0, "dq"), (1, "dk")):
                errs[name] = float((head_norms(mine[:, :, i], 2) / dv).max())
                bars[name] = ZERO_GRAD_BAR
    for k_, err in errs.items():
        assert err < bars[k_], (B, N, H, D, k_, errs)
    o_inf, no_lo, no_lse = K.attn_fwd(qkv.view(-1), B, N, H, D, scale, train=False)
    assert no_lo is None and no_lse is None and torch.equal(o_inf, o)
    return o, lse, dqkv, errs

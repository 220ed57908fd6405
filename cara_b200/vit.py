"""ViT module tree with timm 0.4.12's names and attributes, executed by the cara_b200 CUDA kernels.

The reference builds its backbone with ``timm.models.create_model`` (vit_cp.py:155, tests/test_cara.py:19)
and ``set_cara`` patches timm's ``Attention`` / ``Mlp`` instances (cara.py:147-164).  timm is not a
dependency here: these classes expose the same surface (``blocks[i].{norm1,attn.{qkv,proj,num_heads,scale,
attn_drop,proj_drop},drop_path,norm2,mlp.{fc1,act,fc2,drop}}``, ``patch_embed.proj``, ``cls_token``,
``pos_embed``, ``norm``, ``head``, ``reset_classifier``) and the same 152-key backbone state_dict, so
reference checkpoints load, but every forward runs on the GPU through the C ABI.  There is no CPU forward:
calling a module with CPU tensors raises.
"""
from functools import partial

import torch
import torch.nn as nn

from . import fp32 as F32M
from . import kernels as K
from . import ops
from ._lib import CaraLibraryError

BF16, F32 = torch.bfloat16, torch.float32


def _require_cuda(t, what):
    if not t.is_cuda:
        raise CaraLibraryError(
            "%s: cara_b200 runs on CUDA (sm_100a) only; got a %s tensor -- there is no CPU fallback" % (what, t.device))


class DropPath(nn.Module):
    """Stochastic depth (timm layers/drop.py).  Inside ``VisionTransformer.forward`` the per-sample
    multiplier is folded into the residual add of the next LayerNorm kernel; standalone it scales x."""

    def __init__(self, drop_prob=None):
        super().__init__()
        self.drop_prob = drop_prob

    def rowscale(self, batch, device):
        if not self.training or not self.drop_prob:
            return None
        pre = self.__dict__.get("_predrawn")
        if pre:                                    # drawn for all blocks at once by VisionTransformer.forward
            rs = pre.pop(0)
            if rs.shape[0] == batch and rs.device == device:
                return rs
        keep = 1.0 - self.drop_prob
        return torch.floor(keep + torch.rand(batch, device=device, dtype=F32)) / keep

    def forward(self, x):
        rs = self.rowscale(x.shape[0], x.device)
        return x if rs is None else x * rs.view(-1, *([1] * (x.ndim - 1))).to(x.dtype)


class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        hidden_features = hidden_features or in_features
        out_features = out_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        return mlp_forward(self, x, None)


class Attention(nn.Module):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0.0, proj_drop=0.0):
        super().__init__()
        self.num_heads = num_heads
        self.scale = qk_scale or (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)

    def forward(self, x):
        return attn_forward(self, x, None)


def _as_act(x):
    """[B,N,C] any float dtype -> contiguous bf16 [B*N, C]."""
    B, N, C = x.shape
    return x.reshape(B * N, C).to(BF16).contiguous(), (B, N, C)


def attn_forward(mod, x, staged):
    """Attention branch: fused qkv projection -> attention core -> fused output projection.
    ``staged`` = (qkv terms, proj terms) from ``cara_b200.staging`` or None for the un-adapted module."""
    _require_cuda(x, "Attention.forward")
    if mod.attn_drop.p or mod.proj_drop.p:
        raise NotImplementedError("attn_drop/proj_drop > 0 are not part of the CaRA path (timm default 0)")
    if F32M.is_fp32(mod):
        return F32M.attn_forward(mod, x, staged)
    h, (B, N, C) = _as_act(x)
    H = mod.num_heads
    fq, fp = ops.FrozenLinear.of(mod.qkv), ops.FrozenLinear.of(mod.proj)
    pre, post = mod.__dict__.pop("_cara_rows", None) or (None, None)     # RowsLinks set by Block.fused_step
    if staged is None:
        qkv = ops.CPLinearFunction.apply(h, None, None, None, None, fq, None)
    else:
        A, cs, Bf, _, sink = staged[0].autograd_args()
        qkv = ops.CPLinearFunction.apply(h, A, cs, Bf, None, fq, staged[0].ops, sink, None, pre, None)
    link = ops.AttnLink() if K.attn_delta_fusable(N, C // H) else None
    o = ops.AttnCoreFunction.apply(qkv, B, N, H, C // H, float(mod.scale), link)
    if staged is None:
        y = ops.CPLinearFunction.apply(o, None, None, None, None, fp, None, None, link)
    else:
        A, cs, Bf, bias, sink = staged[1].autograd_args()
        y = ops.CPLinearFunction.apply(o, A, cs, Bf, bias, fp, staged[1].ops, sink, link, None, post)
    y = y.view(B, N, C)
    return y if x.dtype == BF16 else y.to(x.dtype)


def mlp_forward(mod, x, staged):
    """FFN branch: fc1 (+adapter, GELU epilogue) -> fc2 (+adapter)."""
    _require_cuda(x, "Mlp.forward")
    if mod.drop.p:
        raise NotImplementedError("Mlp dropout > 0 is not part of the CaRA path (timm default 0)")
    if not isinstance(mod.act, nn.GELU) or getattr(mod.act, "approximate", "none") != "none":
        raise NotImplementedError("only the exact-erf nn.GELU of timm's Mlp is implemented")
    if F32M.is_fp32(mod):
        return F32M.mlp_forward(mod, x, staged)
    h, (B, N, C) = _as_act(x)
    f1, f2 = ops.FrozenLinear.of(mod.fc1), ops.FrozenLinear.of(mod.fc2)
    pre, post = mod.__dict__.pop("_cara_rows", None) or (None, None)     # RowsLinks set by Block.fused_step
    if staged is None:
        y = ops.CPMlpFunction.apply(h, None, None, None, None, None, None, None, None, f1, None, f2, None)
    else:
        u, d = staged
        a1, c1, b1, bi1, s1 = u.autograd_args()
        a2, c2, b2, bi2, s2 = d.autograd_args()
        y = ops.CPMlpFunction.apply(h, a1, c1, b1, bi1, a2, c2, b2, bi2, f1, u.ops, f2, d.ops, s1, s2, pre, post)
    y = y.view(B, N, -1)
    return y if x.dtype == BF16 else y.to(x.dtype)


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, qk_scale=None, drop=0.0, attn_drop=0.0,
                 drop_path=0.0, act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        # child order matters: set_cara numbers Attention/Mlp instances while walking children()
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop,
                              proj_drop=drop)
        self.drop_path = DropPath(drop_path) if drop_path > 0.0 else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)

    def _rowscale(self, batch, device):
        return self.drop_path.rowscale(batch, device) if isinstance(self.drop_path, DropPath) else None

    def forward(self, x):
        """Stand-alone block (x: [B,N,C]).  ``VisionTransformer.forward`` uses ``fused_step`` instead."""
        _require_cuda(x, "Block.forward")
        B, N, C = x.shape
        xr = x.reshape(B * N, C).to(F32).contiguous()
        h = ops.LayerNormFunction.apply(xr, self.norm1.weight, self.norm1.bias, self.norm1.eps,
                                        F32 if F32M.is_fp32(self) else BF16)
        xr, pending = self.fused_step(xr, h, B, N)
        out = xr + pending[0].float() * (1.0 if pending[1] is None else pending[1].repeat_interleave(N)[:, None])
        return out.view(B, N, C).to(x.dtype)

    def fused_step(self, x, h, B, N, links=None):
        """x fp32 [M,C] residual, h = LN1(x).  Returns (x after the attention add, (mlp branch, rowscale, link))
        with the FFN residual add left pending for the next block's LayerNorm kernel.  ``links`` (from
        ``VisionTransformer._rows_links``) = (qkv forward link -- already filled by the LayerNorm that produced h --,
        fc1 forward link, backward links wanted): the K = C row contractions of the adapter run inside the LayerNorm
        kernels."""
        C = x.shape[1]
        q_fl, f_fl, bwd = links if links is not None else (None, None, False)
        p_bl = ops.RowsLink() if bwd else None                     # proj -> norm2's backward
        m_bl = ops.RowsLink() if bwd else None                     # fc2 -> the next block's norm1 backward
        if links is not None:
            self.attn.__dict__["_cara_rows"] = (q_fl, p_bl)
        a = self.attn(h.view(B, N, C)).reshape(B * N, C)
        self.attn.__dict__.pop("_cara_rows", None)
        x, h2 = ops.AddLayerNormFunction.apply(x, a, self._rowscale(B, x.device), self.norm2.weight,
                                               self.norm2.bias, self.norm2.eps, N, f_fl, p_bl)
        if links is not None:
            self.mlp.__dict__["_cara_rows"] = (f_fl, m_bl)
        m = self.mlp(h2.view(B, N, C)).reshape(B * N, C)
        self.mlp.__dict__.pop("_cara_rows", None)
        return x, (m, self._rowscale(B, x.device), m_bl)


class PatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch_size, patch_size)
        self.grid_size = (img_size // patch_size, img_size // patch_size)
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.norm = nn.Identity()

    def _packed(self):
        w = self.proj.weight
        key = (w.data_ptr(), w._version, w.device)
        cache = self.__dict__.get("_cara_packed")
        if cache is None or cache[0] != key:
            kin = w[0].numel()
            kp = (kin + 63) // 64 * 64
            wm = torch.zeros((w.shape[0], kp), device=w.device, dtype=BF16)
            wm[:, :kin] = w.detach().reshape(w.shape[0], kin).to(BF16)
            cache = (key, wm, kp, self.proj.bias.detach().to(F32).contiguous())
            self.__dict__["_cara_packed"] = cache
        return cache[1], cache[2], cache[3]

    def forward(self, x):
        """[B,3,S,S] fp32 -> bf16 [B, num_patches, C] (im2col + tcgen05 GEMM)."""
        _require_cuda(x, "PatchEmbed.forward")
        if F32M.is_fp32(self):
            return F32M.patch_embed(self, x)
        wm, kp, bias = self._packed()
        patches = K.patchify(x.to(F32).contiguous(), self.patch_size[0], kp)
        return K.gemm_cp(patches, wm, bias=bias).view(x.shape[0], self.num_patches, -1)


def _trunc_normal_(t, std=0.02):
    return nn.init.trunc_normal_(t, std=std, a=-2.0, b=2.0)


class VisionTransformer(nn.Module):
    """timm 0.4.12 ``VisionTransformer`` surface (pre-LN blocks, LN eps 1e-6, class token, learned
    position embedding, Identity pre_logits, Linear head)."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12,
                 num_heads=12, mlp_ratio=4.0, qkv_bias=True, qk_scale=None, drop_rate=0.0, attn_drop_rate=0.0,
                 drop_path_rate=0.0):
        super().__init__()
        self.num_classes = num_classes
        self.num_features = self.embed_dim = embed_dim
        self.num_tokens = 1
        norm_layer = partial(nn.LayerNorm, eps=1e-6)
        self.patch_embed = PatchEmbed(img_size, patch_size, in_chans, embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.patch_embed.num_patches + 1, embed_dim))
        self.pos_drop = nn.Dropout(p=drop_rate)
        rates = [r.item() for r in torch.linspace(0, drop_path_rate, depth)]
        self.blocks = nn.Sequential(*[
            Block(embed_dim, num_heads, mlp_ratio, qkv_bias, qk_scale, drop_rate, attn_drop_rate, rates[i],
                  nn.GELU, norm_layer) for i in range(depth)])
        self.norm = norm_layer(embed_dim)
        self.pre_logits = nn.Identity()
        self.head = nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        _trunc_normal_(self.pos_embed)
        _trunc_normal_(self.cls_token)
        self.apply(self._init_weights)

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            _trunc_normal_(m.weight)
            if m.bias is not None:
                nn.init.zeros_(m.bias)
        elif isinstance(m, nn.LayerNorm):
            nn.init.zeros_(m.bias)
            nn.init.ones_(m.weight)

    def reset_classifier(self, num_classes, global_pool=""):
        self.num_classes = num_classes
        dev = self.cls_token.device
        self.head = (nn.Linear(self.embed_dim, num_classes) if num_classes > 0 else nn.Identity()).to(dev)

    def forward_features(self, img):
        self.__dict__["_cara_fwd_token"] = object()   # one staging of the CP factors per root forward
        try:
            return self._forward_features(img)
        finally:
            self.__dict__["_cara_fwd_token"] = None

    def _forward_features(self, img):
        _require_cuda(img, "VisionTransformer.forward")
        if self.pos_drop.p:
            raise NotImplementedError("pos_drop > 0 is not part of the CaRA path (timm default 0)")
        B = img.shape[0]
        C = self.embed_dim
        N = self.patch_embed.num_patches + 1
        with torch.no_grad():  # everything upstream of block 0 is frozen (vit_cp.py:176-182)
            pe = self.patch_embed(img)
            if F32M.is_fp32(self):   # token assembly is data movement + one add on the frozen path
                x = (torch.cat([self.cls_token.detach().float().expand(B, -1, -1), pe], dim=1)
                     + self.pos_embed.detach().float()).reshape(B * N, C).contiguous()
            else:
                x = K.assemble_tokens(pe.reshape(-1, C), self.cls_token.detach().reshape(C).float().contiguous(),
                                      self.pos_embed.detach().reshape(N, C).float().contiguous(), B, N, C)
        self._predraw_droppath(B, x.device)
        pending = None
        for blk in self.blocks:
            links = self._rows_links(blk)
            q_fl = links[0] if links is not None else None
            if pending is None:
                h = ops.LayerNormFunction.apply(x, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps,
                                                F32 if F32M.is_fp32(self) else BF16, q_fl)
            else:
                x, h = ops.AddLayerNormFunction.apply(x, pending[0], pending[1], blk.norm1.weight, blk.norm1.bias,
                                                      blk.norm1.eps, N, q_fl, pending[2])
            x, pending = blk.fused_step(x, h, B, N, links)
        # only the class-token rows feed the head: finish the last residual add on [B,C]
        xc = x.view(B, N, C)[:, 0]
        if pending is not None:
            d = pending[0].view(B, N, C)[:, 0].float()
            xc = xc + (d if pending[1] is None else d * pending[1][:, None])
        hc = ops.LayerNormFunction.apply(xc.contiguous(), self.norm.weight, self.norm.bias, self.norm.eps, F32)
        return self.pre_logits(hc)

    def _rows_links(self, blk):
        """Forward RowsLinks (qkv, fc1) of one block when the CaRA adapter is installed on this model and its K = C
        row contractions can run inside the LayerNorm kernels (bf16 path, covered (C, Rp), no exact weight dropout)."""
        if not hasattr(self, "CP_A1") or F32M.is_fp32(self) or not hasattr(blk.attn, "attn_idx"):
            return None
        if "forward" not in blk.attn.__dict__ or "forward" not in blk.mlp.__dict__:
            return None                       # un-patched (or merged for --evaluate): the plain forwards take no adapter terms
        from . import staging, wdrop
        if wdrop.wants_exact(self, blk.attn) or wdrop.wants_exact(self, blk.mlp):
            return None
        amap, mmap = staging.staged(self)
        ta, tm = amap.get(id(blk.attn)), mmap.get(id(blk.mlp))
        if ta is None or tm is None or ta[0].ops is None or tm[0].ops is None:
            return None
        rp = ta[0].ops.rp
        fwd, bwd = K.ln_rows_fusable(self.embed_dim, rp), K.ln_rows_fusable(self.embed_dim, rp, backward=True)
        if not (fwd or bwd):
            return None
        train = torch.is_grad_enabled()
        return (ops.RowsLink(ta[0].ops, train) if fwd else None, ops.RowsLink(tm[0].ops, train) if fwd else None, bwd)

    def _predraw_droppath(self, B, device):
        """Stochastic depth draws two per-sample multipliers per block (timm drop_path); draw all of them with
        one rand / add / floor / div instead of four tiny kernels per use."""
        dps = [blk.drop_path for blk in self.blocks if isinstance(blk.drop_path, DropPath)]
        for dp in dps:
            dp.__dict__["_predrawn"] = None
        dps = [dp for dp in dps if dp.training and dp.drop_prob]
        if not dps:
            return
        key = (str(device), tuple(float(dp.drop_prob) for dp in dps))
        cache = self.__dict__.get("_cara_dp_keep")
        if cache is None or cache[0] != key:       # host -> device copy: once, never inside a graph capture
            keep = torch.tensor([1.0 - p for p in key[1] for _ in range(2)], device=device, dtype=F32).view(-1, 1)
            cache = (key, keep)
            self.__dict__["_cara_dp_keep"] = cache
        keep = cache[1]
        rs = torch.floor(keep + torch.rand(keep.shape[0], B, device=device, dtype=F32)) / keep
        for i, dp in enumerate(dps):
            dp.__dict__["_predrawn"] = [rs[2 * i], rs[2 * i + 1]]

    def forward(self, x):
        f = self.forward_features(x)
        if isinstance(self.head, nn.Identity):
            return f
        return ops.HeadFunction.apply(f, self.head.weight, self.head.bias)


_GEOMETRY = {
    "vit_base_patch16_224_in21k": dict(patch_size=16, embed_dim=768, depth=12, num_heads=12, num_classes=21843),
    "vit_base_patch16_224": dict(patch_size=16, embed_dim=768, depth=12, num_heads=12, num_classes=1000),
    "vit_large_patch16_224_in21k": dict(patch_size=16, embed_dim=1024, depth=24, num_heads=16, num_classes=21843),
    "vit_large_patch16_224": dict(patch_size=16, embed_dim=1024, depth=24, num_heads=16, num_classes=1000),
    "vit_huge_patch14_224_in21k": dict(patch_size=14, embed_dim=1280, depth=32, num_heads=16, num_classes=21843),
    # fine-tuned at 384 px (577 tokens): attention runs on the key-tiled kernels of csrc/attention_long.cu
    "vit_base_patch16_384": dict(img_size=384, patch_size=16, embed_dim=768, depth=12, num_heads=12, num_classes=1000),
    "vit_large_patch16_384": dict(img_size=384, patch_size=16, embed_dim=1024, depth=24, num_heads=16, num_classes=1000),
}


def resize_pos_embed(posemb, posemb_new, num_tokens=1, gs_new=()):
    """timm 0.4.12 ``resize_pos_embed``: keep the class-token rows, bilinearly resample the grid rows."""
    import math
    ntok_new = posemb_new.shape[1]
    tok, grid = (posemb[:, :num_tokens], posemb[0, num_tokens:]) if num_tokens else (posemb[:, :0], posemb[0])
    ntok_new -= num_tokens
    gs_old = int(math.sqrt(len(grid)))
    if not len(gs_new):
        gs_new = [int(math.sqrt(ntok_new))] * 2
    grid = grid.reshape(1, gs_old, gs_old, -1).permute(0, 3, 1, 2)
    grid = nn.functional.interpolate(grid, size=tuple(gs_new), mode="bilinear")
    grid = grid.permute(0, 2, 3, 1).reshape(1, gs_new[0] * gs_new[1], -1)
    return torch.cat([tok, grid], dim=1)


@torch.no_grad()
def load_npz_weights(model, checkpoint_path, prefix=""):
    """Import a JAX/Flax ViT checkpoint (``ViT-B_16.npz`` of vit_cp.py:155) into the timm-layout parameters:
    the mapping of timm 0.4.12 ``vision_transformer._load_weights`` (un-vendored dependency, restated) --
    Flax kernels are [in, out] (conv: [P, P, Cin, C]; attention: query/key/value [C, H, D], out [H, D, C]) and
    are transposed into nn.Linear / nn.Conv2d layout; q, k, v are concatenated into ``qkv``; the position
    embedding is resampled when the grid differs; the head is copied only when the class counts agree."""
    import numpy as np

    def n2p(w, t=True):
        if w.ndim == 4 and w.shape[0] == w.shape[1] == w.shape[2] == 1:
            w = w.flatten()
        if t:
            if w.ndim == 4:
                w = w.transpose([3, 2, 0, 1])
            elif w.ndim == 3:
                w = w.transpose([2, 0, 1])
            elif w.ndim == 2:
                w = w.transpose([1, 0])
        return torch.from_numpy(np.ascontiguousarray(w)).float()

    w = np.load(checkpoint_path)
    if not prefix and "opt/target/embedding/kernel" in w:
        prefix = "opt/target/"
    conv = n2p(w[prefix + "embedding/kernel"])
    if conv.shape[1] != model.patch_embed.proj.weight.shape[1]:
        raise ValueError("input channels of the checkpoint (%d) differ from the model's" % conv.shape[1])
    model.patch_embed.proj.weight.copy_(conv)
    model.patch_embed.proj.bias.copy_(n2p(w[prefix + "embedding/bias"]))
    model.cls_token.copy_(n2p(w[prefix + "cls"], t=False))
    pos = n2p(w[prefix + "Transformer/posembed_input/pos_embedding"], t=False)
    if pos.shape != model.pos_embed.shape:
        pos = resize_pos_embed(pos, model.pos_embed, getattr(model, "num_tokens", 1), model.patch_embed.grid_size)
    model.pos_embed.copy_(pos)
    model.norm.weight.copy_(n2p(w[prefix + "Transformer/encoder_norm/scale"]))
    model.norm.bias.copy_(n2p(w[prefix + "Transformer/encoder_norm/bias"]))
    if isinstance(model.head, nn.Linear) and (prefix + "head/bias") in w and \
            model.head.bias.shape[0] == w[prefix + "head/bias"].shape[-1]:
        model.head.weight.copy_(n2p(w[prefix + "head/kernel"]))
        model.head.bias.copy_(n2p(w[prefix + "head/bias"]))
    for i, block in enumerate(model.blocks.children()):
        bp = "%sTransformer/encoderblock_%d/" % (prefix, i)
        mp = bp + "MultiHeadDotProductAttention_1/"
        block.norm1.weight.copy_(n2p(w[bp + "LayerNorm_0/scale"]))
        block.norm1.bias.copy_(n2p(w[bp + "LayerNorm_0/bias"]))
        block.attn.qkv.weight.copy_(torch.cat([n2p(w[mp + n + "/kernel"], t=False).flatten(1).T
                                               for n in ("query", "key", "value")]))
        block.attn.qkv.bias.copy_(torch.cat([n2p(w[mp + n + "/bias"], t=False).reshape(-1)
                                             for n in ("query", "key", "value")]))
        block.attn.proj.weight.copy_(n2p(w[mp + "out/kernel"]).flatten(1))
        block.attn.proj.bias.copy_(n2p(w[mp + "out/bias"]))
        for r in range(2):
            lin = getattr(block.mlp, "fc%d" % (r + 1))
            lin.weight.copy_(n2p(w[bp + "MlpBlock_3/Dense_%d/kernel" % r]))
            lin.bias.copy_(n2p(w[bp + "MlpBlock_3/Dense_%d/bias" % r]))
        block.norm2.weight.copy_(n2p(w[bp + "LayerNorm_2/scale"]))
        block.norm2.bias.copy_(n2p(w[bp + "LayerNorm_2/bias"]))
    return model


def create_model(model_name, pretrained=False, checkpoint_path="", allow_missing_checkpoint=False, **kwargs):
    """``timm.models.create_model`` for the ViT names the reference uses.  ``checkpoint_path``: a JAX ``.npz``
    (vit_cp.py:155, imported by ``load_npz_weights``) or a torch state_dict file.  A missing checkpoint raises, as timm
    does -- fine-tuning a randomly initialised backbone by accident is worse than stopping; synthetic runs (bench,
    tests, ``vit_cp.py --synthetic``) pass ``allow_missing_checkpoint=True`` and keep the random initialisation."""
    if model_name not in _GEOMETRY:
        raise RuntimeError("Unknown model (%s)" % model_name)
    if pretrained:
        raise RuntimeError("pretrained weights need network access; pass checkpoint_path instead")
    cfg = dict(_GEOMETRY[model_name])
    cfg.update(kwargs)
    model = VisionTransformer(**cfg)
    if checkpoint_path:
        import os
        if not os.path.exists(checkpoint_path):
            if not allow_missing_checkpoint:
                raise FileNotFoundError("checkpoint %r not found (pass allow_missing_checkpoint=True / "
                                        "--allow-random-init to keep random-init weights)" % (checkpoint_path,))
            import warnings
            warnings.warn("checkpoint %r not found: keeping random-init weights" % (checkpoint_path,))
        elif str(checkpoint_path).lower().endswith((".npz", ".npy")):
            load_npz_weights(model, checkpoint_path)
        else:
            model.load_state_dict(torch.load(checkpoint_path, map_location="cpu"), strict=False)
    return model

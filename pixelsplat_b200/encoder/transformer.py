"""Transformer building blocks with the reference's parameter tree
(/root/reference/src/model/transformer/{attention,transformer,pre_norm,feed_forward}.py), so that
reference checkpoints load with strict=True (SURVEY.md Appendix C).

`Attention.forward(x, z)` accepts, besides a tensor `z`, an `EpipolarKV` handle: the keys/values
are then never materialised -- the fused CUDA kernel gathers them from the feature map
(pixelsplat_b200/encoder/attention_fused.py).  If a forward hook is registered on `attend` (the
reference's visualisers hook `transformer.layers[i][0].fn.attend`,
encoder_visualizer_epipolar.py:53-56) the module falls back to the explicit soft-max path so the
hook sees the [(b v r), head, 1, s*ov] attention tensor it expects.  It takes the same explicit path for
shapes the kernel does not cover (more than 4 heads or 32 samples, features other than 128 channels,
a depth encoding wider than the kernel's; `attention_fused.supported`), which the reference accepts.

With z = None (ImageSelfAttention's ViT blocks) and the shape the kernel is written for (256 tokens,
128-dim heads) the soft-max attention runs on the tcgen05 tensor cores
(pixelsplat_b200/encoder/self_attention_tc.py); other shapes use torch's fp32 matmul + softmax.
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from . import self_attention_tc as _satc
from .attention_fused import EpipolarKV, fused_epipolar_attention, fused_supported


class Attention(nn.Module):
    def __init__(self, dim, heads=8, dim_head=64, dropout=0.0, selfatt=True, kv_dim=None):
        super().__init__()
        inner_dim = dim_head * heads
        project_out = not (heads == 1 and dim_head == dim)
        self.heads = heads
        self.dim_head = dim_head
        self.scale = dim_head ** -0.5
        self.attend = nn.Softmax(dim=-1)
        if selfatt:
            self.to_qkv = nn.Linear(dim, inner_dim * 3, bias=False)
        else:
            self.to_q = nn.Linear(dim, inner_dim, bias=False)
            self.to_kv = nn.Linear(kv_dim, inner_dim * 2, bias=False)
        self.to_out = (nn.Sequential(nn.Linear(inner_dim, dim), nn.Dropout(dropout))
                       if project_out else nn.Identity())

    def _split(self, t: Tensor) -> Tensor:
        b, n, _ = t.shape
        return t.reshape(b, n, self.heads, self.dim_head).transpose(1, 2)

    def forward(self, x: Tensor, z=None) -> Tensor:
        if isinstance(z, EpipolarKV):
            hooked = len(self.attend._forward_hooks) > 0 or len(self.attend._forward_pre_hooks) > 0
            if not hooked and isinstance(self.to_out, nn.Sequential) and fused_supported(self, z):
                return fused_epipolar_attention(self, x, z)
            z = z.materialize()
        if z is None:
            qkv = self.to_qkv(x)
            hooked = len(self.attend._forward_hooks) > 0 or len(self.attend._forward_pre_hooks) > 0
            if not hooked and _satc.supported(qkv, self.heads, self.dim_head):
                # dense per-image self-attention on the tensor cores (csrc/self_attention_tc.cu)
                return self.to_out(_satc.self_attention_tc(qkv, self.heads, self.scale))
            q, k, v = qkv.chunk(3, dim=-1)
        else:
            q = self.to_q(x)
            k, v = self.to_kv(z).chunk(2, dim=-1)
        q, k, v = self._split(q), self._split(k), self._split(v)
        attn = self.attend(torch.matmul(q, k.transpose(-1, -2)) * self.scale)
        out = torch.matmul(attn, v).transpose(1, 2)
        out = out.reshape(out.shape[0], out.shape[1], self.heads * self.dim_head)
        return self.to_out(out)


class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim, dropout=0.0):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden_dim), nn.GELU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, dim), nn.Dropout(dropout))

    def forward(self, x):
        return self.net(x)


class PreNorm(nn.Module):
    """LayerNorm on x only (never on the context z), as the reference's pre_norm.py:34-35."""

    def __init__(self, dim, fn):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn

    def forward(self, x, **kwargs):
        return self.fn(self.norm(x), **kwargs)


class Transformer(nn.Module):
    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout=0.0, selfatt=True, kv_dim=None,
                 feed_forward_layer=FeedForward):
        super().__init__()
        self.layers = nn.ModuleList([])
        for _ in range(depth):
            self.layers.append(nn.ModuleList([
                PreNorm(dim, Attention(dim, heads=heads, dim_head=dim_head, dropout=dropout,
                                       selfatt=selfatt, kv_dim=kv_dim)),
                PreNorm(dim, feed_forward_layer(dim, mlp_dim, dropout=dropout)),
            ]))

    def forward(self, x, z=None, **kwargs):
        for attn, ff in self.layers:
            x = attn(x, z=z) + x
            x = ff(x, **kwargs) + x
        return x

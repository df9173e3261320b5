"""Host side of the fused epipolar cross-attention: the `EpipolarKV` handle that stands in for the
reference's materialised key/value tensor, the autograd Function over the C ABI
(`ps_epipolar_attention_forward/backward`), and the weight folding around it.

Reference semantics being reproduced: /root/reference/src/model/transformer/attention.py:54-70 with
z = sampling.features + depth_encoding(+ view embeddings)
(/root/reference/src/model/encoder/epipolar/epipolar_transformer.py:103-142).  See
csrc/epipolar_attention.cu for the algebra.  All dense projections stay torch GEMMs, so autograd
delivers the gradients of to_q / to_kv / to_out / depth_encoding / view_embeddings unchanged.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Optional

import torch
from torch import Tensor

from .. import _lib


def _p(t: Optional[Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


@dataclass
class EpipolarGeometry:
    """Output of ps_epipolar_geometry for one forward (shared by every layer)."""
    segments: Tensor       # [b, v, ov, r, 4]  xy_min.xy, xy_max.xy (masked, NaN-free)
    valid: Tensor          # [b, v, ov, r] uint8
    rel_disparity: Tensor  # [b, v, ov, r, s]
    t_range: Tensor        # [b, v, ov, r, 2]
    grid: tuple[int, int]  # (h, w) of the ray grid
    samples: int


def epipolar_geometry(extrinsics: Tensor, intrinsics: Tensor, near: Tensor, far: Tensor,
                      grid: tuple[int, int], samples: int) -> EpipolarGeometry:
    if not extrinsics.is_cuda:
        raise ValueError("extrinsics must be a CUDA tensor (pixelsplat_b200 has no CPU path)")
    b, v = extrinsics.shape[:2]
    h, w = grid
    ov, r = v - 1, h * w
    dev = extrinsics.device
    f = lambda t: t.to(torch.float32).contiguous()
    e, k, nr, fr = f(extrinsics), f(intrinsics), f(near), f(far)
    seg = torch.empty((b, v, ov, r, 4), dtype=torch.float32, device=dev)
    valid = torch.empty((b, v, ov, r), dtype=torch.uint8, device=dev)
    rd = torch.empty((b, v, ov, r, samples), dtype=torch.float32, device=dev)
    tr = torch.empty((b, v, ov, r, 2), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    rc = _lib.on_device(dev, _lib.lib.ps_epipolar_geometry, b, v, h, w, samples, _p(e), _p(k), _p(nr), _p(fr), _p(seg), _p(valid),
                                       _p(rd), _p(tr), ctypes.c_void_p(stream.cuda_stream))
    _lib.check(rc, "ps_epipolar_geometry")
    return EpipolarGeometry(seg, valid, rd, tr, (h, w), samples)


class EpipolarKV:
    """What `Transformer.forward(q, z=...)` receives instead of the [(b v r), (s ov), c] tensor."""

    def __init__(self, features: Tensor, geometry: EpipolarGeometry, depth_linear, pe_module,
                 view_embeddings: Optional[Tensor]):
        # features: [b, v, c, h, w] (the down-scaled maps the samples are drawn from)
        self.features = features
        self.features_cl = features.permute(0, 1, 3, 4, 2).contiguous()   # channels-last, autograd-tracked
        self.geometry = geometry
        self.depth_linear = depth_linear        # nn.Linear(2*octaves, c) or None
        self.pe_module = pe_module              # PositionalEncoding or None
        self.view_embeddings = view_embeddings  # [ov, c] (already permuted) or None

    # ---- explicit path (hooks / debugging): builds exactly the reference's kv tensor
    def sample_features(self) -> Tensor:
        """[b, v, ov, r, s, c] = bilinear samples * valid (epipolar_sampler.py:97-111)."""
        import torch.nn.functional as F
        g = self.geometry
        b, v, c, h, w = self.features.shape
        ov, r, s = v - 1, h * w, g.samples
        u = (torch.arange(s, device=self.features.device, dtype=torch.float32) + 0.5) / s
        lo, hi = g.segments[..., None, :2], g.segments[..., None, 2:]
        xy = lo + u[:, None] * (hi - lo)                               # [b, v, ov, r, s, 2]
        out = []
        for vi in range(v):
            per_ov = []
            for o in range(ov):
                other = o if o < vi else o + 1
                grid = (2 * xy[:, vi, o] - 1).reshape(b, r * s, 1, 2)
                smp = F.grid_sample(self.features[:, other], grid, mode="bilinear", padding_mode="zeros",
                                    align_corners=False)               # [b, c, r*s, 1]
                per_ov.append(smp[..., 0].permute(0, 2, 1).reshape(b, r, s, c))
            out.append(torch.stack(per_ov, 1))
        feats = torch.stack(out, 1)
        return feats * g.valid[..., None, None].to(feats.dtype)

    def materialize(self) -> Tensor:
        g = self.geometry
        kv = self.sample_features()
        if self.depth_linear is not None:
            kv = kv + self.depth_linear(self.pe_module(g.rel_disparity[..., None]))
        if self.view_embeddings is not None:
            kv = kv + self.view_embeddings[None, None, :, None, None, :]
        b, v, ov, r, s, c = kv.shape
        return kv.permute(0, 1, 3, 4, 2, 5).reshape(b * v * r, s * ov, c)   # "(b v r) (s ov) c"


def supported(heads: int, channels: int, samples: int, pe_dim: int, views: int) -> bool:
    """Whether the fused kernel takes this shape: the checks of `epi_check` (csrc/epipolar_attention.cu)."""
    return (1 <= heads <= 4 and channels == 128 and 1 <= samples <= 32 and 0 <= pe_dim <= 32
            and pe_dim % 2 == 0 and heads * pe_dim <= 96 and 2 <= views <= 33)


def fused_supported(attn, kv: EpipolarKV) -> bool:
    """`supported` for the `Attention` module `attn` attending to `kv`."""
    pe_dim = 0 if kv.depth_linear is None else kv.depth_linear.in_features
    return supported(attn.heads, kv.features.shape[2], kv.geometry.samples, pe_dim, kv.features.shape[1])


class _EpipolarAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qt, pq, bias, feat_cl, geometry: EpipolarGeometry, heads: int):
        if not feat_cl.is_cuda:
            raise ValueError("pixelsplat_b200 has no CPU path: the epipolar attention needs CUDA tensors")
        b, v, h, w, c = feat_cl.shape
        n = b * v * h * w
        dev = feat_cl.device
        npe = pq.shape[-1]
        desc = _lib.EpipolarDesc(b, v, h, w, geometry.samples, c, heads, npe)
        qt, pq = qt.contiguous(), pq.contiguous()
        bias_c = None if bias is None else bias.contiguous()
        inputs = _lib.EpipolarInputs(feat_cl.data_ptr(), geometry.segments.data_ptr(),
                                     geometry.valid.data_ptr(), geometry.rel_disparity.data_ptr(),
                                     qt.data_ptr(), pq.data_ptr(),
                                     None if bias_c is None else bias_c.data_ptr())
        z = torch.empty((n, heads, c), dtype=torch.float32, device=dev)
        e = torch.empty((n, heads, npe), dtype=torch.float32, device=dev)
        mass = torch.empty((n, heads, v - 1), dtype=torch.float32, device=dev)
        lse = torch.empty((n, heads), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev)
        rc = _lib.on_device(dev, _lib.lib.ps_epipolar_attention_forward, ctypes.byref(desc), ctypes.byref(inputs), _p(z), _p(e),
                                                    _p(mass), _p(lse), ctypes.c_void_p(stream.cuda_stream))
        _lib.check(rc, "ps_epipolar_attention_forward")
        ctx.save_for_backward(qt, pq, bias_c if bias_c is not None else torch.empty(0, device=dev), feat_cl,
                              z, e, mass, lse)
        ctx.geometry, ctx.desc, ctx.has_bias = geometry, desc, bias_c is not None
        return z, e, mass

    @staticmethod
    def backward(ctx, dz, de, dmass):
        qt, pq, bias, feat_cl, z, e, mass, lse = ctx.saved_tensors
        g, desc = ctx.geometry, ctx.desc
        dev = feat_cl.device
        dz, de = dz.contiguous().float(), de.contiguous().float()
        use_mass = dmass is not None          # mass is an output with or without a bias input
        d_row = (dz * z).sum(-1) + (de * e).sum(-1)
        if use_mass:
            dmass = dmass.contiguous().float()
            d_row = d_row + (dmass * mass).sum(-1)
        d_row = d_row.contiguous()
        inputs = _lib.EpipolarInputs(feat_cl.data_ptr(), g.segments.data_ptr(), g.valid.data_ptr(),
                                     g.rel_disparity.data_ptr(), qt.data_ptr(), pq.data_ptr(),
                                     bias.data_ptr() if ctx.has_bias else None)
        dqt = torch.empty_like(qt)
        dpq = torch.empty_like(pq)
        dbias = torch.empty_like(bias) if ctx.has_bias else None
        dfeat = torch.zeros_like(feat_cl)
        stream = torch.cuda.current_stream(dev)
        rc = _lib.on_device(dev, _lib.lib.ps_epipolar_attention_backward,
            ctypes.byref(desc), ctypes.byref(inputs), _p(lse), _p(dz), _p(de), _p(dmass) if use_mass else None,
            _p(d_row), _p(dqt), _p(dpq), _p(dbias), _p(dfeat), ctypes.c_void_p(stream.cuda_stream))
        _lib.check(rc, "ps_epipolar_attention_backward")
        return dqt, dpq, dbias, dfeat, None, None


def fused_epipolar_attention(attn, x: Tensor, kv: EpipolarKV) -> Tensor:
    """attn: the `Attention` module (to_q / to_kv / to_out); x: [n, 1, c] (already layer-normed).
    The shape must pass `fused_supported(attn, kv)`."""
    n, one, c = x.shape
    assert one == 1
    H, d = attn.heads, attn.dim_head
    wq = attn.to_q.weight.reshape(H, d, c)                # [H, d, c_in]
    wk, wv = attn.to_kv.weight.reshape(2, H, d, -1).unbind(0)   # [H, d, c_kv]
    wo = attn.to_out[0].weight.reshape(-1, H, d)          # [c_out, H, d]
    bo = attn.to_out[0].bias
    # qt_h = scale * W_k,h^T W_q,h x   (one GEMM with the folded [H*c_kv, c_in] matrix)
    a = torch.einsum("hdk,hde->hke", wk, wq) * attn.scale              # [H, c_kv, c_in]
    xin = x[:, 0]
    qt = (xin @ a.reshape(H * a.shape[1], c).t()).reshape(n, H, -1)    # [n, H, c_kv]
    if kv.depth_linear is not None:
        wd, bd = kv.depth_linear.weight, kv.depth_linear.bias         # [c_kv, npe], [c_kv]
        pq = qt @ wd                                                   # [n, H, npe]
    else:
        wd = bd = None
        pq = torch.zeros((n, H, 0), dtype=x.dtype, device=x.device)
    bias = None
    if kv.view_embeddings is not None:
        bias = qt @ kv.view_embeddings.t()                             # [n, H, ov]
    z, e, mass = _EpipolarAttentionFn.apply(qt, pq, bias, kv.features_cl, kv.geometry, H)
    kvbar = z
    if wd is not None:
        kvbar = kvbar + e @ wd.t() + bd
    if kv.view_embeddings is not None:
        kvbar = kvbar + mass @ kv.view_embeddings
    # y = sum_h W_o,h W_v,h kvbar_h + b_o   (one GEMM with the folded [c_out, H*c_kv] matrix)
    u = torch.einsum("ohd,hdk->ohk", wo, wv)                           # [c_out, H, c_kv]
    y = kvbar.reshape(n, -1) @ u.reshape(u.shape[0], -1).t() + bo
    y = attn.to_out[1](y)                                              # dropout (p = 0 in pixelSplat)
    return y[:, None]

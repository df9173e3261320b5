"""The fused epipolar attention kernels (csrc/epipolar_attention.cu, `k_epi_attn_fwd` / `k_epi_attn_bwd`) against a
float64 statement of their contract, at the shapes, optional inputs and segment geometries the C ABI accepts.

`epipolar_contract` below is that statement: exactly what include/pixelsplat_b200.h promises for
ps_epipolar_attention_forward, as plain torch.  The CPU test `test_contract_reproduces_the_explicit_path` shows
that, substituted for the kernel, it makes the module's weight folding reproduce the reference's explicit path
(materialised K/V, torch soft-max) to 1e-10 in float64, so the contract is the reference's semantics.

Bars (fixed from the arithmetic before any GPU run; "own" is the error of the SAME contract evaluated in float32
torch on the CPU, where no TF32 can enter, against float64):
  z / e / mass   max-norm relative error <= max(4 own, 2e-6), capped at 2e-5
  lse            |delta| <= 2e-5 max(1, |lse|)
  gradients      tests.util.grad_errors: l2 <= max(4 own, 1e-6) capped at 1e-4, and max <= 1e-3
The kernel forms each score from a 128-term float32 dot product plus a <= 32-term PE dot product and runs the
soft-max online (rescales cost one rounding each), like the float32 evaluation; its positional encoding is more
accurate than float32 torch's (exact phase reduction), so at 10+ octaves "own" is large and the cap decides.
Each case prints ours / own per quantity.
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
import sys
from dataclasses import dataclass
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import golden_util as gu
from tests.util import grad_errors, rel_err

ROOT = Path(__file__).resolve().parents[1]
GOLD = ROOT / "tests" / "golden"
DEV = "cuda:0"
C = 128
# the reference's PositionalEncoding buffers are float32: frequency float32(2 pi) 2^k, phases (0, float32(pi / 2))
TWO_PI_F32 = float(torch.tensor(2 * math.pi, dtype=torch.float32))
PHASES = (0.0, float(torch.tensor(0.5 * math.pi, dtype=torch.float32)))


# ---------------------------------------------------------------------------------------------------------------
# the contract
# ---------------------------------------------------------------------------------------------------------------

def epipolar_contract(feat, seg, valid, rd, qt, pq, bias, dtype=torch.float64, scores=False):
    """ps_epipolar_attention_forward in plain torch.

    feat [B, V, h, w, 128], seg [B, V, OV, R, 4] (xy_min, xy_max), valid [B, V, OV, R], rd [B, V, OV, R, S],
    qt [N, H, 128], pq [N, H, npe], bias [N, H, OV] or None, with N = B V R and query n = (b V + v) R + r.
    Returns z [N, H, 128], e [N, H, npe], mass [N, H, OV], lse [N, H] in `dtype` (and the scores if asked).
    Sample positions are formed in float32 from the float32 segment, as the kernel does; everything after that
    is `dtype`.  Rays with valid = 0 contribute zero features (their segment is never read) but keep their PE."""
    B, V, h, w, c = feat.shape
    OV, R, S = V - 1, h * w, rd.shape[-1]
    H, npe = qt.shape[1], pq.shape[-1]
    dev = feat.device
    u = (torch.arange(S, device=dev, dtype=torch.float32) + 0.5) / S
    seg32 = seg.to(torch.float32)
    lo, hi = seg32[..., None, :2], seg32[..., None, 2:]
    xy = lo + u[:, None] * (hi - lo)                                        # [B, V, OV, R, S, 2]
    ok = valid.to(torch.bool)
    xy = torch.where(ok[..., None, None], xy, torch.zeros_like(xy)).to(dtype)
    other = torch.tensor([[o if o < v else o + 1 for o in range(OV)] for v in range(V)], device=dev)
    maps = feat.to(dtype)[:, other].reshape(B * V * OV, h, w, c).permute(0, 3, 1, 2)
    grid = (2 * xy - 1).reshape(B * V * OV, R * S, 1, 2)
    f = F.grid_sample(maps, grid, mode="bilinear", padding_mode="zeros", align_corners=False)
    f = f[..., 0].permute(0, 2, 1).reshape(B, V, OV, R, S, c) * ok[..., None, None].to(dtype)
    k = torch.arange(npe // 2, device=dev, dtype=dtype)
    phase = torch.tensor(PHASES, device=dev, dtype=dtype)
    pe = torch.sin((rd.to(dtype)[..., None] * (TWO_PI_F32 * 2.0 ** k))[..., None] + phase).flatten(-2)
    q = qt.to(dtype).reshape(B, V, R, H, c)
    p = pq.to(dtype).reshape(B, V, R, H, npe)
    sc = torch.einsum("bvrhc,bvorsc->bvrhos", q, f) + torch.einsum("bvrhj,bvorsj->bvrhos", p, pe)
    if bias is not None:
        sc = sc + bias.to(dtype).reshape(B, V, R, H, OV)[..., None]
    flat = sc.reshape(B, V, R, H, OV * S)
    lse = torch.logsumexp(flat, -1)
    a = torch.exp(flat - lse[..., None]).reshape(sc.shape)
    z = torch.einsum("bvrhos,bvorsc->bvrhc", a, f)
    e = torch.einsum("bvrhos,bvorsj->bvrhj", a, pe)
    mass = a.sum(-1)
    N = B * V * R
    out = (z.reshape(N, H, c), e.reshape(N, H, npe), mass.reshape(N, H, OV), lse.reshape(N, H))
    return out + (sc,) if scores else out


# ---------------------------------------------------------------------------------------------------------------
# CPU: the contract is the reference's semantics
# ---------------------------------------------------------------------------------------------------------------

def _dyadic_geometry(b, v, h, w, S, gen):
    """CPU geometry whose sample positions are exact in float32 AND float64 (segment ends k / 64, S = 32), so
    the explicit path (which forms them in the segments' dtype) and the contract (float32) see the same points."""
    from pixelsplat_b200.encoder.attention_fused import EpipolarGeometry
    ov, r = v - 1, h * w
    seg = torch.randint(-16, 81, (b, v, ov, r, 4), generator=gen).double() / 64
    valid = (torch.rand(b, v, ov, r, generator=gen) > 0.2).to(torch.uint8)
    rd = torch.rand(b, v, ov, r, S, generator=gen).float()
    return EpipolarGeometry(seg, valid, rd, torch.zeros(b, v, ov, r, 2), (h, w), S)


@pytest.mark.parametrize("octaves", [10, 0])
@pytest.mark.parametrize("v", [2, 3])
def test_contract_reproduces_the_explicit_path(v, octaves, monkeypatch):
    """With `epipolar_contract` in place of the kernel, `fused_epipolar_attention`'s folding (qt = scale W_k^T W_q x,
    pq = qt W_d, bias = qt emb^T, then the W_o W_v unfold) equals the explicit path -- materialise() and the torch
    soft-max, forced by a hook on `attend` -- in float64 to 1e-10, output and every gradient."""
    from pixelsplat_b200.encoder import EpipolarTransformer, EpipolarTransformerCfg, ImageSelfAttentionCfg
    from pixelsplat_b200.encoder import attention_fused as af
    cfg = EpipolarTransformerCfg(ImageSelfAttentionCfg(4, 10, 2, 4, 128, 128, 256), octaves, 2, 4, 32, 128, 256, 4)
    m = EpipolarTransformer(cfg, 128, num_context_views=v)
    gu.fill_parameters(m)
    m = m.double()
    gen = torch.Generator().manual_seed(17 * v + octaves)
    b, h, w, S = 1, 3, 5, 32
    geom = _dyadic_geometry(b, v, h, w, S, gen)
    feats = torch.randn(b, v, C, h, w, generator=gen, dtype=torch.float64).requires_grad_(True)
    x = torch.randn(b * v * h * w, 1, C, generator=gen, dtype=torch.float64).requires_grad_(True)
    attn = m.transformer.layers[0][0].fn
    depth_linear = m.depth_encoding[1] if octaves else None
    pe_module = m.depth_encoding[0] if octaves else None

    def run(explicit):
        emb = m.view_embeddings(torch.tensor([1, 0])) if v > 2 else None
        kv = af.EpipolarKV(feats, geom, depth_linear, pe_module, emb)
        hook = attn.attend.register_forward_hook(lambda *a: None) if explicit else None
        try:
            y = attn(x, z=kv)
        finally:
            if hook is not None:
                hook.remove()
        wgt = torch.randn(y.shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
        params = [x, feats] + [p for p in m.parameters()]
        grads = torch.autograd.grad((y * wgt).sum(), params, allow_unused=True)
        return y.detach(), grads

    # the product has no CPU path: unpatched, the fold reaches the autograd Function, which refuses CPU tensors
    with pytest.raises(ValueError, match="no CPU path"):
        run(False)
    calls = []

    def contract_apply(qt, pq, bias, feat_cl, g, heads):
        calls.append(heads)
        z, e, mass, _ = epipolar_contract(feat_cl, g.segments, g.valid, g.rel_disparity, qt, pq, bias)
        return z, e, mass

    monkeypatch.setattr(af._EpipolarAttentionFn, "apply", contract_apply)
    y_f, g_f = run(False)
    assert calls == [4]
    y_e, g_e = run(True)
    assert calls == [4]
    assert rel_err(y_f.numpy(), y_e.numpy()) <= 1e-10
    for gf, ge in zip(g_f, g_e):
        assert (gf is None) == (ge is None)
        if gf is not None:
            assert rel_err(gf.numpy(), ge.numpy()) <= 1e-10


def test_no_depth_fixtures_are_usable():
    """The num_octaves = 0 goldens (oracle/make_epipolar_golden.py, the reference's no-depth-encoding ablation):
    each under 1 MB, no depth_encoding entries, and the reference's own float32 error small enough that the
    module bar (2x own, <= 5e-3) is meaningful."""
    for v in (2, 3):
        path = GOLD / f"epipolar_transformer_no_depth_v{v}.npz"
        assert path.stat().st_size < 1 << 20
        gold = np.load(path)
        assert not any("depth_encoding" in k for k in gold.files)
        assert ("f64_grad:view_embeddings.weight" in gold.files) == (v > 2)
        for key in ("core", "out_sub", "dfeat_sub"):
            assert rel_err(gold["f32_" + key].astype(np.float64), gold["f64_" + key]) < 1e-3, key


# ---------------------------------------------------------------------------------------------------------------
# ABI argument validation (no launch happens, so this runs without a GPU too)
# ---------------------------------------------------------------------------------------------------------------

def test_abi_rejects_unsupported_shapes_before_any_launch():
    from pixelsplat_b200 import _lib
    dev = DEV if torch.cuda.is_available() else "cpu"
    # buffers large enough for every descriptor below, so no launch could leave them even if a check were missing
    buf = torch.zeros(1 << 20, device=dev)
    ptr = ctypes.c_void_p(buf.data_ptr())
    good = dict(batch=1, views=2, grid_h=2, grid_w=2, samples=4, channels=128, heads=2, pe_dim=4)
    full = lambda: _lib.EpipolarInputs(*[buf.data_ptr()] * 7)
    bad = [("heads", 0, 3, "heads"), ("heads", 5, 3, "heads"), ("samples", 0, 3, "samples"),
           ("samples", 33, 3, "samples"), ("pe_dim", 3, 3, "pe_dim"), ("pe_dim", 34, 3, "pe_dim"),
           ("channels", 64, 3, "channels"), ("views", 1, 1, "views"), ("views", 34, 3, "33 views")]
    cases = [(dict(good, **{k: val}), rc, msg) for k, val, rc, msg in bad]
    cases.append((dict(good, heads=4, pe_dim=26), 3, "pe_dim"))          # heads * pe_dim = 104 > 96
    for kw, want_rc, msg in cases:
        d = _lib.EpipolarDesc(**kw)
        for fn, args in ((_lib.lib.ps_epipolar_attention_forward, [ptr] * 4 + [None]),
                         (_lib.lib.ps_epipolar_attention_backward, [ptr] * 9 + [None])):
            rc = fn(ctypes.byref(d), ctypes.byref(full()), *args)
            assert rc == want_rc, (kw, rc)
            assert msg.encode() in _lib.lib.ps_last_error(), (kw, _lib.lib.ps_last_error())
    d = _lib.EpipolarDesc(**good)
    for field in ("features", "segments", "valid", "rel_disparity", "q_feat", "q_pe"):
        inp = full()
        setattr(inp, field, None)
        assert _lib.lib.ps_epipolar_attention_forward(ctypes.byref(d), ctypes.byref(inp), ptr, ptr, ptr, ptr, None) == 1
        assert b"NULL" in _lib.lib.ps_last_error()
        assert _lib.lib.ps_epipolar_attention_backward(ctypes.byref(d), ctypes.byref(inp), *[ptr] * 9, None) == 1
        assert b"NULL" in _lib.lib.ps_last_error()
    fwd_outs = [ptr] * 4
    for i in (0, 1, 3):                                                    # z, e, lse (mass may be NULL)
        outs = list(fwd_outs)
        outs[i] = None
        assert _lib.lib.ps_epipolar_attention_forward(ctypes.byref(d), ctypes.byref(full()), *outs, None) == 1
        assert b"NULL" in _lib.lib.ps_last_error()
    for i in (0, 1, 2, 4, 5, 6, 8):                        # lse, dz, de, d_row, dq_feat, dq_pe, dfeatures
        outs = [ptr] * 9
        outs[i] = None
        assert _lib.lib.ps_epipolar_attention_backward(ctypes.byref(d), ctypes.byref(full()), *outs, None) == 1
        assert b"NULL" in _lib.lib.ps_last_error()


# ---------------------------------------------------------------------------------------------------------------
# GPU: kernel vs float64
# ---------------------------------------------------------------------------------------------------------------

KINDS = ("inside", "cross", "band_left", "band_bottom", "outside", "far", "zero", "reversed", "texel", "centre",
         "nan", "invalid")


def _segment(kind, r, h, w, g):
    """One segment (x0, y0, x1, y1) and its valid flag."""
    rnd = lambda lo, hi: float(lo + (hi - lo) * torch.rand((), generator=g, dtype=torch.float64))
    if kind == "inside":
        return [rnd(.05, .95) for _ in range(4)], 1
    if kind == "cross":                # leaves the map through the left and the bottom edge
        return [rnd(.2, .8), rnd(.2, .8), rnd(-.4, -.05), rnd(1.05, 1.4)], 1
    if kind == "band_left":            # inside the half-texel band x in (-0.5 / w, 0.5 / w)
        return [-0.49 / w, rnd(.1, .9), 0.49 / w, rnd(.1, .9)], 1
    if kind == "band_bottom":          # y in (1 - 0.5 / h, 1 + 0.5 / h), reversed
        return [rnd(.1, .9), 1 + 0.49 / h, rnd(.1, .9), 1 - 0.49 / h], 1
    if kind == "outside":              # valid, but every tap is padding
        return [rnd(-2, -1.1), rnd(-1, 2), rnd(-2, -1.1), rnd(-1, 2)], 1
    if kind == "far":                  # wild coordinates (clamped before the int cast), all outside
        return [-1e3, 5e2, -40.0, -3e2], 1
    if kind == "zero":                 # zero length: every sample in one bilinear cell
        x, y = rnd(.05, .95), rnd(.05, .95)
        return [x, y, x, y], 1
    if kind == "reversed":
        return [rnd(.6, .95), rnd(.6, .95), rnd(.05, .4), rnd(.05, .4)], 1
    if kind == "texel":                # zero length on a texel centre (ax = ay = 0)
        x, y = ((r * 7) % w + 0.5) / w, ((r * 3) % h + 0.5) / h
        return [x, y, x, y], 1
    if kind == "centre":               # through the texel centres of a row (samples on centres when S = w)
        y = (r % h + 0.5) / h
        return [0.0, y, 1.0, y], 1
    if kind == "nan":                  # an invalid ray: its segment must never be read
        return [float("nan")] * 4, 0
    return [rnd(.05, .95) for _ in range(4)], 0          # "invalid" with a finite segment


@dataclass(frozen=True)
class Case:
    name: str
    B: int
    V: int
    h: int
    w: int
    S: int
    H: int
    npe: int
    bias: bool = True
    qscale: float = 0.1
    kinds: tuple = KINDS
    same_view: bool = False        # view 0: every ray (each b, each other view) has one and the same segment


CASES = [
    Case("h1_S1_pe32_v3_5x9", 1, 3, 5, 9, 1, 1, 32),
    Case("h2_S2_pe2_v2_B2_1x7_nobias", 2, 2, 1, 7, 2, 2, 2, bias=False),
    Case("h3_S3_pe32_v3_7x1", 1, 3, 7, 1, 3, 3, 32),
    Case("h4_S4_pe24_v5_5x9", 1, 5, 5, 9, 4, 4, 24),
    Case("h4_S5_pe20_v3_B2_1x1_nobias", 2, 3, 1, 1, 5, 4, 20, bias=False),
    Case("h2_S7_pe0_v2_16x16", 1, 2, 16, 16, 7, 2, 0, bias=False),
    Case("h1_S8_pe20_v33_1x7", 1, 33, 1, 7, 8, 1, 20),
    Case("h3_S9_pe2_v3_B2_5x9_same", 2, 3, 5, 9, 9, 3, 2, same_view=True),
    Case("h4_S13_pe20_v5_7x1_nobias", 1, 5, 7, 1, 13, 4, 20, bias=False),
    Case("h4_S16_pe20_v2_16x16_centres", 1, 2, 16, 16, 16, 4, 20, bias=False, kinds=("centre", "texel")),
    Case("h4_S31_pe24_v3_5x9", 1, 3, 5, 9, 31, 4, 24),
    Case("h4_S32_pe20_v3_B2_16x16_same", 2, 3, 16, 16, 32, 4, 20, same_view=True),
    Case("h2_S32_pe0_v33_1x1_nobias", 1, 33, 1, 1, 32, 2, 0, bias=False),
    Case("h3_S32_pe32_v2_5x9", 1, 2, 5, 9, 32, 3, 32, bias=False),
    Case("scores60_h4_S13_pe20_v3_5x9", 1, 3, 5, 9, 13, 4, 20, qscale=3.0, kinds=("inside", "reversed", "cross")),
]
SUB4_SUBSET = ("h1_S1_", "h3_S3_", "h4_S5_", "h3_S9_", "h4_S13_", "h4_S31_", "h1_S8_", "scores60")


def make_inputs(case: Case, seed: int = 0):
    """CPU tensors of one case: geometry by hand, features, folded queries and output cotangents."""
    g = torch.Generator().manual_seed(seed + sum(map(ord, case.name)))
    B, V, h, w, S, H, npe = case.B, case.V, case.h, case.w, case.S, case.H, case.npe
    OV, R = V - 1, h * w
    seg = torch.empty(B, V, OV, R, 4, dtype=torch.float32)
    valid = torch.empty(B, V, OV, R, dtype=torch.uint8)
    for b in range(B):
        for v in range(V):
            for o in range(OV):
                for r in range(R):
                    kind = case.kinds[(r + 3 * o + 5 * v + 7 * b) % len(case.kinds)]
                    sg, ok = _segment(kind, r, h, w, g)
                    seg[b, v, o, r] = torch.tensor(sg)
                    valid[b, v, o, r] = ok
    if case.same_view:
        seg[:, 0] = torch.tensor([0.31, 0.42, 0.38, 0.47])
        valid[:, 0] = 1
    rd = torch.rand(B, V, OV, R, S, generator=g)
    ridx = torch.arange(R)
    rd[..., ridx % 5 == 1, :] = 0.0
    rd[..., ridx % 5 == 2, :] = 1.0
    N = B * V * R
    rnd = lambda *shape, s=1.0: torch.randn(*shape, generator=g) * s
    return dict(feat=rnd(B, V, h, w, C), seg=seg, valid=valid, rd=rd, qt=rnd(N, H, C, s=case.qscale),
                pq=rnd(N, H, npe, s=0.3), bias=rnd(N, H, OV, s=0.5) if case.bias else None,
                dz=rnd(N, H, C), de=rnd(N, H, npe), dmass=rnd(N, H, OV))


def _geometry(inp, S, dev=DEV):
    from pixelsplat_b200.encoder.attention_fused import EpipolarGeometry
    B, V, h, w, _ = inp["feat"].shape
    return EpipolarGeometry(inp["seg"].to(dev).contiguous(), inp["valid"].to(dev).contiguous(),
                            inp["rd"].to(dev).contiguous(), None, (h, w), S)


def run_contract(inp, dtype, dev="cpu", mass_grad=True):
    """The contract and its autograd gradients (of sum dz.z + de.e + dmass.mass) in `dtype` on `dev`."""
    t = {k: (None if v is None else v.to(dev)) for k, v in inp.items()}
    leaves = {k: t[k].to(dtype).requires_grad_(True) for k in ("qt", "pq", "feat") + (("bias",) if t["bias"] is not None else ())}
    z, e, mass, lse = epipolar_contract(leaves["feat"], t["seg"], t["valid"], t["rd"], leaves["qt"], leaves["pq"],
                                        leaves.get("bias"), dtype=dtype)
    loss = (z * t["dz"].to(dtype)).sum() + (e * t["de"].to(dtype)).sum()
    if mass_grad:
        loss = loss + (mass * t["dmass"].to(dtype)).sum()
    grads = dict(zip(leaves, torch.autograd.grad(loss, list(leaves.values()))))
    out = dict(z=z, e=e, mass=mass, lse=lse)
    return ({k: v.detach().cpu().double() for k, v in out.items()},
            {"d" + k: v.cpu().double() for k, v in grads.items()})


def bar_scales(inp):
    """(cap scale, floor scale) of one input set; see the module docstring."""
    *_, sc = epipolar_contract(*[inp[k] for k in ("feat", "seg", "valid", "rd", "qt", "pq", "bias")], scores=True)
    B, V, OV, R, S = inp["rd"].shape
    return max(1.0, float(sc.abs().max()) / 10), max(1.0, math.sqrt(OV * S / 256))


def run_kernel(inp, H, S):
    """Forward and backward through `_EpipolarAttentionFn` (the module's entry to the C ABI)."""
    from pixelsplat_b200.encoder.attention_fused import _EpipolarAttentionFn
    t = {k: (None if v is None else v.to(DEV)) for k, v in inp.items()}
    leaves = {k: t[k].clone().requires_grad_(True) for k in ("qt", "pq", "feat") + (("bias",) if t["bias"] is not None else ())}
    z, e, mass = _EpipolarAttentionFn.apply(leaves["qt"], leaves["pq"], leaves.get("bias"), leaves["feat"],
                                            _geometry(inp, S), H)
    lse = z.grad_fn.saved_tensors[7]
    loss = (z * t["dz"]).sum() + (e * t["de"]).sum() + (mass * t["dmass"]).sum()
    grads = dict(zip(leaves, torch.autograd.grad(loss, list(leaves.values()))))
    torch.cuda.synchronize()
    out = dict(z=z, e=e, mass=mass, lse=lse)
    return ({k: v.detach().cpu().double() for k, v in out.items()},
            {"d" + k: v.cpu().double() for k, v in grads.items()})


FWD_FLOOR, FWD_CAP, LSE_TOL = 2e-6, 2e-5, 2e-5
GRAD_FLOOR, GRAD_CAP, GRAD_MAX = 1e-6, 1e-4, 1e-3


def check_against_contract(name, ours, own, ref, ours_g=None, own_g=None, ref_g=None, scales=(1.0, 1.0)):
    """Asserts the bars of the module docstring (`scales` from `bar_scales`); prints ours / own per quantity."""
    report, failures = {}, []
    cap_s, floor_s = scales
    for k in ("z", "e", "mass"):
        if ref[k].numel() == 0:
            continue
        o, w_ = rel_err(ours[k].numpy(), ref[k].numpy()), rel_err(own[k].numpy(), ref[k].numpy())
        bar = min(max(4 * w_, FWD_FLOOR * floor_s), FWD_CAP * cap_s)
        report[k] = (o, w_)
        if not (np.isfinite(ours[k].numpy()).all() and o <= bar):
            failures.append((k, o, w_, bar))
    dl = (ours["lse"] - ref["lse"]).abs() / ref["lse"].abs().clamp(min=1.0)
    report["lse"] = (float(dl.max()), float(((own["lse"] - ref["lse"]).abs() / ref["lse"].abs().clamp(min=1.0)).max()))
    if not (torch.isfinite(ours["lse"]).all() and float(dl.max()) <= LSE_TOL * cap_s):
        failures.append(("lse", float(dl.max()), LSE_TOL))
    for k in (ref_g or {}):
        if ref_g[k].numel() == 0:
            continue
        o, w_ = grad_errors(ours_g[k].numpy(), ref_g[k].numpy()), grad_errors(own_g[k].numpy(), ref_g[k].numpy())
        bar = min(max(4 * w_["l2"], GRAD_FLOOR * floor_s), GRAD_CAP * cap_s)
        report[k] = (o["l2"], w_["l2"])
        if not (np.isfinite(ours_g[k].numpy()).all() and o["l2"] <= bar and o["max"] <= GRAD_MAX):
            failures.append((k, o, w_["l2"], bar))
    print(f"{name}: " + ", ".join(f"{k} {a:.1e}/{b:.1e}" for k, (a, b) in report.items()) + "  (ours/own)")
    assert not failures, (name, failures)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_kernel_matches_float64(case):
    inp = make_inputs(case)
    ours, ours_g = run_kernel(inp, case.H, case.S)
    ref, ref_g = run_contract(inp, torch.float64)
    own, own_g = run_contract(inp, torch.float32)
    check_against_contract(case.name, ours, own, ref, ours_g, own_g, ref_g, bar_scales(inp))
    if case.qscale > 1:
        # the score-range case does what it says: scores spread over about +-60 and one sample carries most weight
        _, _, _, _, sc = epipolar_contract(*[inp[k] for k in ("feat", "seg", "valid", "rd", "qt", "pq", "bias")],
                                           scores=True)
        flat = sc.flatten(-2)
        assert float((flat.amax(-1) - flat.amin(-1)).median()) > 60
        assert float(torch.softmax(flat, -1).amax(-1).median()) > 0.9


@pytest.mark.gpu
def test_optional_mass_and_dmass_may_be_null():
    """Direct ABI calls: forward with mass = NULL, backward with dmass = NULL (d_row then has no mass term)."""
    from pixelsplat_b200 import _lib
    case = Case("nullable_h3_S9_pe20_v5_5x9", 1, 5, 5, 9, 9, 3, 20)
    inp = make_inputs(case)
    t = {k: (None if v is None else v.to(DEV).contiguous()) for k, v in inp.items()}
    B, V, h, w, S, H, npe = case.B, case.V, case.h, case.w, case.S, case.H, case.npe
    N, OV = B * V * h * w, V - 1
    p = lambda x: None if x is None else ctypes.c_void_p(x.data_ptr())
    desc = _lib.EpipolarDesc(B, V, h, w, S, C, H, npe)
    inputs = _lib.EpipolarInputs(*[t[k].data_ptr() for k in ("feat", "seg", "valid", "rd", "qt", "pq", "bias")])
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    nan = lambda *s: torch.full(s, float("nan"), device=DEV)
    z, e, lse = nan(N, H, C), nan(N, H, npe), nan(N, H)
    _lib.check(_lib.lib.ps_epipolar_attention_forward(ctypes.byref(desc), ctypes.byref(inputs), p(z), p(e), None,
                                                      p(lse), stream), "forward")
    d_row = ((t["dz"] * z).sum(-1) + (t["de"] * e).sum(-1)).contiguous()
    dqt, dpq, dbias, dfeat = nan(N, H, C), nan(N, H, npe), nan(N, H, OV), torch.zeros_like(t["feat"])
    _lib.check(_lib.lib.ps_epipolar_attention_backward(
        ctypes.byref(desc), ctypes.byref(inputs), p(lse), p(t["dz"]), p(t["de"]), None, p(d_row), p(dqt), p(dpq),
        p(dbias), p(dfeat), stream), "backward")
    torch.cuda.synchronize()
    ref, ref_g = run_contract(inp, torch.float64, mass_grad=False)
    own, own_g = run_contract(inp, torch.float32, mass_grad=False)
    ours = dict(z=z.cpu().double(), e=e.cpu().double(), mass=ref["mass"], lse=lse.cpu().double())
    ours_g = dict(dqt=dqt.cpu().double(), dpq=dpq.cpu().double(), dbias=dbias.cpu().double(),
                  dfeat=dfeat.cpu().double())
    check_against_contract(case.name, ours, own, ref, ours_g, own_g, ref_g, bar_scales(inp))


@pytest.mark.gpu
def test_zero_scores_give_the_plain_mean():
    """qt = pq = bias = 0: every score is 0, so z is the plain mean of the OV S samples, mass = 1 / OV and
    lse = log(OV S).  Samples sit on texel centres (S = w, segments through a row's centres) and rd = 0, so the
    samples are texel values and PE = (0, 1, 0, 1, ...): the answer needs no reference."""
    from pixelsplat_b200.encoder.attention_fused import _EpipolarAttentionFn
    B, V, h, w, H, npe = 2, 3, 4, 8, 2, 4
    OV, R, S = V - 1, h * w, w
    case = Case("zero", B, V, h, w, S, H, npe, kinds=("centre",))
    inp = make_inputs(case)
    inp["rd"].zero_()
    feat = inp["feat"].to(DEV)
    z, e, mass = _EpipolarAttentionFn.apply(torch.zeros(B * V * R, H, C, device=DEV, requires_grad=True),
                                            torch.zeros(B * V * R, H, npe, device=DEV),
                                            torch.zeros(B * V * R, H, OV, device=DEV), feat, _geometry(inp, S), H)
    lse = z.grad_fn.saved_tensors[7]
    z, e, mass = z.detach(), e.detach(), mass.detach()
    f64 = inp["feat"].double()
    want = torch.empty(B, V, R, C, dtype=torch.float64)
    for b in range(B):
        for v in range(V):
            others = [o if o < v else o + 1 for o in range(OV)]
            for r in range(R):
                want[b, v, r] = f64[b, others][:, r % h].mean((0, 1))
    want = want.reshape(B * V * R, 1, C).expand(-1, H, -1)
    assert rel_err(z.cpu().double().numpy(), want.numpy()) < 1e-6
    assert torch.allclose(mass.cpu(), torch.full((B * V * R, H, OV), 1.0 / OV), rtol=0, atol=1e-6)
    assert torch.allclose(lse.cpu(), torch.full((B * V * R, H), math.log(OV * S)), rtol=0, atol=2e-5 * math.log(OV * S))
    want_e = torch.tensor([0.0, 1.0] * (npe // 2)).expand(B * V * R, H, npe)
    assert torch.allclose(e.cpu(), want_e, rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_config2_shaped_layer_matches_float64():
    """One layer at the configs[2] shape: B = 2, V = 2, 64 x 64 rays, S = 32, 4 heads, pe_dim 20, geometry from
    epipolar_geometry() on the generic rig.  The float64 contract runs on the GPU (TF32 off for its duration)."""
    from pixelsplat_b200.encoder.attention_fused import epipolar_geometry
    B, V, h, w, S, H, npe = 2, 2, 64, 64, 32, 4, 20
    ext, K, near, far = [t.to(DEV, torch.float32) for t in gu.camera_rig(B, V, "generic")]
    geom = epipolar_geometry(ext, K, near, far, (h, w), S)
    case = Case("config2", B, V, h, w, S, H, npe, bias=False)
    g = torch.Generator().manual_seed(2)
    N, OV = B * V * h * w, V - 1
    rnd = lambda *shape, s=1.0: torch.randn(*shape, generator=g) * s
    inp = dict(feat=rnd(B, V, h, w, C), seg=geom.segments.cpu(), valid=geom.valid.cpu(), rd=geom.rel_disparity.cpu(),
               qt=rnd(N, H, C, s=0.1), pq=rnd(N, H, npe, s=0.3), bias=None, dz=rnd(N, H, C), de=rnd(N, H, npe),
               dmass=rnd(N, H, OV))
    assert 0.2 < float(geom.valid.float().mean()) < 1.0
    ours, ours_g = run_kernel(inp, H, S)
    tf32_conv, tf32_mm = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref, ref_g = run_contract(inp, torch.float64, dev=DEV)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32_conv, tf32_mm
    own, own_g = run_contract(inp, torch.float32)
    check_against_contract(case.name, ours, own, ref, ours_g, own_g, ref_g, bar_scales(inp))


@pytest.mark.gpu
def test_sub4_forward_variant_matches_float64():
    """The forward's 4-sample sub-chunk variant (PIXELSPLAT_B200_EPI_SUB_FWD=4, read once per process) on a
    subset of the cases above covering every S mod 4 remainder, in a child process that ends with the test."""
    if os.environ.get("PIXELSPLAT_B200_EPI_SUB_FWD"):
        pytest.skip("already running the selected variant")
    env = dict(os.environ, PIXELSPLAT_B200_EPI_SUB_FWD="4")
    sel = " or ".join(SUB4_SUBSET)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", str(Path(__file__)), "-q", "-s", "-p", "no:cacheprovider", "-m", "gpu",
        "-k", f"test_kernel_matches_float64 and ({sel})"]
    r = subprocess.run(cmd, cwd=str(ROOT), env=env, capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert f"{len(SUB4_SUBSET)} passed" in r.stdout


# ---------------------------------------------------------------------------------------------------------------
# GPU: module level -- unsupported shapes fall back, supported shapes keep the kernel
# ---------------------------------------------------------------------------------------------------------------

def _module(octaves=10, heads=4, samples=32, d_in=128, v=2):
    from pixelsplat_b200.encoder import EpipolarTransformer, EpipolarTransformerCfg, ImageSelfAttentionCfg
    cfg = EpipolarTransformerCfg(ImageSelfAttentionCfg(4, 10, 2, 4, 128, 128, 256), octaves, 2, heads, samples, 128,
                                 256, 4)
    m = EpipolarTransformer(cfg, d_in, num_context_views=v)
    gu.fill_parameters(m)
    return m.to(DEV)


def _counting_apply(monkeypatch):
    from pixelsplat_b200.encoder import attention_fused as af
    calls, orig = [], af._EpipolarAttentionFn.apply

    def counted(*args):
        calls.append(args[-1])
        return orig(*args)

    monkeypatch.setattr(af._EpipolarAttentionFn, "apply", counted)
    return calls


def _step(m, d_in, v, explicit=False):
    ext, K, near, far = [t.to(DEV, torch.float32) for t in gu.camera_rig(1, v, "generic")]
    feats = gu.seeded_like("features", (1, v, d_in, 32, 32), 1.0, torch.float32).to(DEV).requires_grad_(True)
    wgt = gu.seeded_like("loss_weight", (1, v, d_in, 32, 32), 1.0, torch.float32).to(DEV)
    hooks = ([layer[0].fn.attend.register_forward_hook(lambda *a: None) for layer in m.transformer.layers]
             if explicit else [])
    m.zero_grad()
    torch.manual_seed(0)
    out, _ = m(feats, ext, K, near, far)
    (out * wgt).sum().backward()
    for hk in hooks:
        hk.remove()
    return out.detach(), feats.grad, {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(heads=8), dict(samples=48), dict(octaves=13), dict(d_in=64)],
                         ids=["heads8", "samples48", "octaves13", "d_in64"])
def test_unsupported_shapes_fall_back_to_the_explicit_path(kw, monkeypatch):
    """Shapes the reference accepts but the kernel does not: forward and backward run (no PS_ERR_UNSUPPORTED),
    never call the kernel, equal the explicit path, and an optimiser step trains."""
    calls = _counting_apply(monkeypatch)
    d_in = kw.get("d_in", 128)
    m = _module(**kw)
    out, gfeat, grads = _step(m, d_in, 2)
    assert calls == []
    out_e, gfeat_e, grads_e = _step(m, d_in, 2, explicit=True)
    # the bars of test_epipolar_gpu.py::test_fused_attention_equals_explicit_path (atomic reductions in grid_sample's
    # backward and cuDNN make two runs of one path differ by ~1e-5 already)
    assert rel_err(out.cpu().numpy(), out_e.cpu().numpy()) < 1e-3
    assert rel_err(gfeat.cpu().numpy(), gfeat_e.cpu().numpy()) < 2e-3
    assert grads.keys() == grads_e.keys()
    for n in grads:
        assert torch.isfinite(grads[n]).all() and rel_err(grads[n].cpu().numpy(), grads_e[n].cpu().numpy()) < 3e-3, n
    opt = torch.optim.SGD(m.parameters(), lr=1e-3)
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    opt.step()
    assert any(not torch.equal(before[n], p) for n, p in m.named_parameters())


@pytest.mark.gpu
@pytest.mark.parametrize("octaves,v", [(10, 2), (10, 3), (0, 2), (0, 3)])
def test_supported_shapes_use_the_kernel(octaves, v, monkeypatch):
    """The reference config and its num_octaves = 0 ablation keep the fused kernel: once per layer."""
    calls = _counting_apply(monkeypatch)
    m = _module(octaves=octaves, v=v)
    out, gfeat, _ = _step(m, 128, v)
    assert calls == [4, 4]
    assert torch.isfinite(out).all() and torch.isfinite(gfeat).all()

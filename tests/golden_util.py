"""Deterministic inputs/weights shared by oracle/make_epipolar_golden.py (which runs the REFERENCE
modules in this container) and the tests (which run the drop-in on the GPU box, where
/root/reference does not exist).  Nothing is stored for inputs or weights: both sides regenerate
them from these rules; only reference OUTPUTS live in tests/golden/*.npz."""
from __future__ import annotations

import math
import zlib

import torch


def load_npz_refs(*paths) -> dict:
    """np.load of the fixtures of one recording, merged, whose writer stored byte-identical large arrays once
    (`key__ref` names the first copy; oracle/make_render_args_golden.py)."""
    import numpy as np
    raws = [np.load(p) for p in paths]
    out = {k: raw[k] for raw in raws for k in raw.files if not k.endswith("__ref")}
    for raw in raws:
        for k in raw.files:
            if k.endswith("__ref"):
                out[k[:-5]] = out[str(raw[k])]
    return out


def seeded_like(name: str, shape, scale: float = 1.0, dtype=torch.float64) -> torch.Tensor:
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    return (torch.randn(tuple(shape), generator=g, dtype=torch.float64) * scale).to(dtype)


def fill_parameters(module: torch.nn.Module) -> None:
    """Name-keyed deterministic parameters (independent of construction order / RNG state)."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if p.dim() > 1:
                fan_in = p[0].numel()
                v = seeded_like(name, p.shape, 1.0 / math.sqrt(fan_in))
            elif name.endswith("norm.weight"):
                v = 1.0 + seeded_like(name, p.shape, 0.1)
            else:
                v = seeded_like(name, p.shape, 0.1)
            p.copy_(v.to(p.dtype))


def rotation(rx: float, ry: float, rz: float) -> torch.Tensor:
    cx, sx, cy, sy, cz, sz = (math.cos(rx), math.sin(rx), math.cos(ry), math.sin(ry), math.cos(rz), math.sin(rz))
    Rx = torch.tensor([[1, 0, 0], [0, cx, -sx], [0, sx, cx]], dtype=torch.float64)
    Ry = torch.tensor([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]], dtype=torch.float64)
    Rz = torch.tensor([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]], dtype=torch.float64)
    return Rz @ Ry @ Rx


def camera_rig(b: int, v: int, case: str = "generic"):
    """Deterministic camera-to-world extrinsics [b,v,4,4], normalised intrinsics [b,v,3,3],
    near/far [b,v] (float64).  Cases exercise the edge rules of project_rays / intersect_rays:
      generic   views spread along x with small rotations (the re10k situation)
      parallel  identical orientation and identical position for two views (parallel rays -> 1e10)
      diverging cameras looking away from each other (most rays miss the other image: invalid)
    """
    ext = torch.eye(4, dtype=torch.float64).repeat(b, v, 1, 1)
    K = torch.eye(3, dtype=torch.float64).repeat(b, v, 1, 1)
    for bi in range(b):
        for vi in range(v):
            s = 0.37 * bi + 0.91 * vi
            if case == "generic":
                ext[bi, vi, :3, :3] = rotation(0.03 * math.sin(s), 0.08 * math.cos(2 * s) * vi, 0.02 * math.sin(3 * s))
                ext[bi, vi, :3, 3] = torch.tensor([1.0 * vi / max(v - 1, 1), 0.05 * math.sin(s), 0.04 * math.cos(s)],
                                                   dtype=torch.float64)
            elif case == "parallel":
                ext[bi, vi, :3, 3] = torch.tensor([0.0 if vi < 2 else 0.5, 0.0, 0.0], dtype=torch.float64)
            elif case == "diverging":
                ext[bi, vi, :3, :3] = rotation(0.0, (1.2 if vi % 2 else -1.2), 0.0)
                ext[bi, vi, :3, 3] = torch.tensor([0.3 * vi, 0.0, 0.0], dtype=torch.float64)
            f = 0.88 + 0.03 * math.sin(1.7 * s)
            K[bi, vi, 0, 0], K[bi, vi, 1, 1] = f, f * 1.02
            K[bi, vi, 0, 2], K[bi, vi, 1, 2] = 0.5 + 0.01 * math.cos(s), 0.5 - 0.01 * math.sin(s)
    near = torch.full((b, v), 0.293, dtype=torch.float64) * (1 + 0.1 * torch.arange(v, dtype=torch.float64))
    far = torch.full((b, v), 450.6, dtype=torch.float64)
    return ext, K, near, far


def adapter_case(b: int = 2, v: int = 2, r: int = 40, srf: int = 1, spp: int = 3, d_sh: int = 25, case: str = "generic"):
    """Inputs of GaussianAdapter.forward in EncoderEpipolar's call shape (float64): extrinsics
    [b,v,1,1,1,4,4], intrinsics [b,v,1,1,1,3,3], coordinates [b,v,r,srf,1,2] in (0,1), depths and
    opacities [b,v,r,srf,spp], raw [b,v,r,srf,1,7+3 d_sh], plus loss weights for every output."""
    ext, K, near, far = camera_rig(b, v, case)
    lead = (b, v, r, srf, spp)
    coords = torch.sigmoid(seeded_like("adapter.coords", (b, v, r, srf, 1, 2)))
    u = torch.sigmoid(seeded_like("adapter.depth", lead))
    depths = 1.0 / ((1 - u) * (1 / near - 1 / far)[:, :, None, None, None] + (1 / far)[:, :, None, None, None])
    opac = torch.sigmoid(seeded_like("adapter.opacity", lead)) / spp
    raw = seeded_like("adapter.raw", (b, v, r, srf, 1, 7 + 3 * d_sh))
    weights = {k: seeded_like("adapter.w." + k, shape) for k, shape in dict(
        means=(*lead, 3), covariances=(*lead, 3, 3), harmonics=(*lead, 3, d_sh), scales=(*lead, 3),
        rotations=(*lead, 4), opacities=lead).items()}
    return dict(extrinsics=ext[:, :, None, None, None], intrinsics=K[:, :, None, None, None], coordinates=coords,
                depths=depths, opacities=opac, raw=raw, near=near, far=far, weights=weights)


def adapter_loss(g, weights) -> torch.Tensor:
    """A scalar that touches every output of the adapter (covariances weighted up: they are ~1e-4)."""
    return ((g.means * weights["means"]).sum() + 1e3 * (g.covariances * weights["covariances"]).sum()
            + (g.harmonics * weights["harmonics"]).sum() + 10.0 * (g.scales * weights["scales"]).sum()
            + (g.rotations * weights["rotations"]).sum() + (g.opacities * weights["opacities"]).sum())

"""Generates tests/golden/render_cuda_args.npz by running the REFERENCE's own host code --
`render_cuda`, `render_depth_cuda`, `render_cuda_orthographic`
(/root/reference/src/model/decoder/cuda_splatting.py:47-269, unmodified) -- on the CPU with a
RECORDING stand-in for its rasterizer extension (SURVEY.md 8c "fake backend").  Authoring container only:

    python oracle/make_render_args_golden.py

TEST INFRASTRUCTURE.  The reference's `diff_gaussian_rasterization` dependency is un-vendored, so the only
thing of the rasterizer boundary that CAN be pinned to the reference is what the reference's host code
hands to it: the `GaussianRasterizationSettings` it builds (image size, tan(fov) python floats, bg,
transposed = column-major view / full-projection matrices, stride-4 `campos`, sh_degree, flags) and the
tensors of `GaussianRasterizer.forward` (means3D, zero means2D, `[P, M, 3]` shs or `[P, 3]`
colors_precomp, `[P, 1]` opacities, `[P, 6]` triu covariances).  The recorder stores exactly those, per
view, together with the scene that produced them.  Tests then check
  * CPU: the oracle's restatement of that host code (oracle/raster_torch.prepare_view, which every
    rasterizer parity test builds its arguments with) reproduces the recorded arguments;
  * GPU: the recorded arguments through the drop-in `GaussianRasterizer` give the same image as
    `pixelsplat_b200.decoder.render_cuda` on the scene, and `ps_camera_setup` reproduces the matrices.
"""
from __future__ import annotations

import sys
import types
from pathlib import Path
from typing import NamedTuple

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import epipolar_ref  # noqa: E402
from pixelsplat_b200 import synthetic  # noqa: E402

OUT = ROOT / "tests" / "golden"
RECORDS: list[dict] = []


class GaussianRasterizationSettings(NamedTuple):      # the extension's NamedTuple, field for field
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


class GaussianRasterizer(torch.nn.Module):
    """Records what it is called with; returns a constant image so the caller's stacking code runs."""

    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None,
                rotations=None, cov3D_precomp=None):
        rs = self.raster_settings
        rec = dict(
            image_height=int(rs.image_height), image_width=int(rs.image_width),
            tanfovx=float(rs.tanfovx), tanfovy=float(rs.tanfovy), scale_modifier=float(rs.scale_modifier),
            sh_degree=int(rs.sh_degree), prefiltered=bool(rs.prefiltered), debug=bool(rs.debug),
            campos_stride=int(rs.campos.stride(0)), campos_contiguous=bool(rs.campos.is_contiguous()),
            viewmatrix_contiguous=bool(rs.viewmatrix.is_contiguous()),
            bg=rs.bg.detach().clone(), viewmatrix=rs.viewmatrix.detach().clone(),
            projmatrix=rs.projmatrix.detach().clone(), campos=rs.campos.detach().clone(),
            means3D=means3D.detach().clone(), means2D=means2D.detach().clone(),
            means2D_requires_grad=bool(means2D.requires_grad), opacities=opacities.detach().clone(),
            shs=None if shs is None else shs.detach().clone(),
            colors_precomp=None if colors_precomp is None else colors_precomp.detach().clone(),
            cov3D_precomp=cov3D_precomp.detach().clone(), has_scales=scales is not None,
            has_rotations=rotations is not None)
        RECORDS.append(rec)
        h, w = rs.image_height, rs.image_width
        return torch.zeros((3, h, w), dtype=means3D.dtype), torch.zeros(means3D.shape[0], dtype=torch.int32)


def load_reference_cuda_splatting():
    epipolar_ref.load(2)                                   # sys.path + bare `src.model.encoder` / `src.dataset`
    stub = types.ModuleType("diff_gaussian_rasterization")
    stub.GaussianRasterizationSettings = GaussianRasterizationSettings
    stub.GaussianRasterizer = GaussianRasterizer
    sys.modules["diff_gaussian_rasterization"] = stub
    if "src.model.decoder" not in sys.modules:             # skip decoder/__init__ (imports the dataset package)
        m = types.ModuleType("src.model.decoder")
        m.__path__ = [str(epipolar_ref.REFERENCE / "src/model/decoder")]
        sys.modules["src.model.decoder"] = m
    from src.model.decoder import cuda_splatting
    return cuda_splatting


def scene():
    """Two target cameras over their own copies of a small re10k-like scene (render_cuda's call shape:
    every batch element brings its Gaussians), float32."""
    sc = synthetic.scene_re10k_like(seed=77, image_hw=(16, 16), target_views=2)
    b = sc.extrinsics.shape[0]
    rep = lambda t: t[None].expand(b, *t.shape).contiguous()
    ext = sc.extrinsics.clone()
    # give the second camera a rotation so the matrices are not axis-aligned
    c, s = np.cos(0.07), np.sin(0.07)
    ext[1, :3, :3] = ext[1, :3, :3] @ torch.tensor([[c, 0, s], [0, 1, 0], [-s, 0, c]], dtype=torch.float32)
    return dict(extrinsics=ext, intrinsics=sc.intrinsics.clone(), near=sc.near.clone(), far=sc.far.clone(),
                means=rep(sc.means), covariances=rep(sc.covariances), harmonics=rep(sc.harmonics),
                opacities=rep(sc.opacities), background=torch.tensor([[0.0, 0.0, 0.0], [0.1, 0.2, 0.3]]),
                image_shape=(24, 40))


_SEEN: dict[bytes, str] = {}


def store(out: dict, key: str, value) -> None:
    """Large arrays that are byte-identical to one already stored (the same Gaussians reach the rasterizer
    in several calls) are stored once; `key__ref` then names the first copy (tests/golden_util.load_npz_refs)."""
    a = value.numpy() if torch.is_tensor(value) else np.asarray(value)
    if a.nbytes >= 4096:
        h = a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()
        if h in _SEEN:
            out[key + "__ref"] = np.asarray(_SEEN[h])
            return
        _SEEN[h] = key
    out[key] = a


def take(prefix: str, out: dict) -> None:
    for i, rec in enumerate(RECORDS):
        for k, v in rec.items():
            if v is not None:
                store(out, f"{prefix}_{i}_{k}", v)
    out[f"{prefix}_n"] = np.asarray(len(RECORDS))
    RECORDS.clear()


def main():
    cs = load_reference_cuda_splatting()
    s = scene()
    # the scene goes to render_cuda_scene.npz, the recorded calls to render_cuda_args.npz (each file under 1 MB)
    scene_out = {}
    for k, v in s.items():
        store(scene_out, f"scene_{k}", v[:1] if k in ("means", "covariances", "harmonics", "opacities") else v)
    out = {}
    args = (s["extrinsics"], s["intrinsics"], s["near"], s["far"], s["image_shape"])
    g = (s["means"], s["covariances"], s["harmonics"], s["opacities"])
    img = cs.render_cuda(*args, s["background"], *g)
    assert img.shape == (2, 3, 24, 40)
    take("render_cuda", out)
    cs.render_cuda(*args, s["background"], *g, scale_invariant=False)
    take("render_cuda_noscale", out)
    for mode in ("depth", "disparity", "relative_disparity", "log"):
        d = cs.render_depth_cuda(*args, s["means"], s["covariances"], s["opacities"], mode=mode)
        assert d.shape == (2, 24, 40)
        take(f"render_depth_{mode}", out)
    # the reference's orthographic path only runs at batch 1 (`move_back[2, 3] = -distance_to_near`, :164,
    # needs a one-element tensor), which is how validation_in_3d.py:68 calls it
    dump = {}
    ortho_ext = torch.eye(4)[None].clone()
    ortho_ext[:, 2, 3] = -1.0
    c, sn = np.cos(0.3), np.sin(0.3)
    ortho_ext[0, :3, :3] = torch.tensor([[c, 0, sn], [0, 1, 0], [-sn, 0, c]], dtype=torch.float32)
    out["ortho_extrinsics"] = ortho_ext.numpy()
    out["ortho_width"] = np.asarray([2.0], np.float32)
    out["ortho_height"] = np.asarray([2.5], np.float32)
    out["ortho_near"] = np.asarray([0.0], np.float32)
    out["ortho_far"] = np.asarray([50.0], np.float32)
    cs.render_cuda_orthographic(ortho_ext, torch.tensor(out["ortho_width"]), torch.tensor(out["ortho_height"]),
                                torch.tensor(out["ortho_near"]), torch.tensor(out["ortho_far"]), s["image_shape"],
                                s["background"][1:], *[t[:1] for t in g], dump=dump)
    take("render_ortho", out)
    for k, v in dump.items():
        out[f"ortho_dump_{k}"] = v.numpy()
    assert all(np.array_equal(s[k][0].numpy(), s[k][1].numpy()) for k in ("means", "covariances", "harmonics", "opacities"))
    # get_projection_matrix on its own (cuda_splatting.py:17-44)
    fov = torch.tensor([[0.9, 0.7], [1.2, 1.1]])
    out["proj_fov"] = fov.numpy()
    out["proj_matrix"] = cs.get_projection_matrix(s["near"], s["far"], fov[:, 0], fov[:, 1]).numpy()
    OUT.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(OUT / "render_cuda_scene.npz", **scene_out)
    np.savez_compressed(OUT / "render_cuda_args.npz", **out)
    print("wrote", OUT / "render_cuda_args.npz", len(out), "arrays;",
          {k: out[k].shape for k in ("render_cuda_0_shs", "render_cuda_0_cov3D_precomp", "render_cuda_0_viewmatrix")},
          "campos stride", out["render_cuda_0_campos_stride"])


if __name__ == "__main__":
    main()

"""GPU tests against tests/golden/render_cuda_args.npz (the arguments the REFERENCE's own render_cuda /
render_depth_cuda / render_cuda_orthographic hand to their rasterizer, recorded by
oracle/make_render_args_golden.py): rows a1 / a2 / a5 / a6 / b1 pinned to the reference's host code.

  * the recorded per-view arguments, fed through the drop-in `diff_gaussian_rasterization` classes exactly
    as the reference would (`GaussianRasterizationSettings(...)`, `GaussianRasterizer(settings)(...)`),
    must give the image that `pixelsplat_b200.decoder.render_*` gives on the scene itself (batched launch,
    native layouts, fused rescale, device-side camera set-up) -- and both must agree with the CPU oracle
    evaluated on the recorded arguments;
  * `ps_camera_setup` must reproduce the recorded matrices / tan(fov) / campos to float32 round-off.
Tolerances: images as in tests/test_raster_gpu.py (>= 99.5 % of pixels within 2e-5, PSNR > 60 dB: the two
paths build their matrices with different float32 operation orders, so a Gaussian may flip a tile or a
1/255 decision); matrices 2e-6 relative to the largest entry.
"""
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import golden_util as gu
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = Path(__file__).resolve().parent / "golden"
G = gu.load_npz_refs(GOLD / "render_cuda_args.npz", GOLD / "render_cuda_scene.npz")
H, W = 24, 40


def T(k):
    return torch.from_numpy(np.asarray(G[k])).to(DEV)


def _scene(n=2):
    s = {k: T(f"scene_{k}") for k in ("extrinsics", "intrinsics", "near", "far", "background")}
    for k in ("means", "covariances", "harmonics", "opacities"):
        s[k] = T(f"scene_{k}").expand(n, *G[f"scene_{k}"].shape[1:]).contiguous()
    return s


def _dropin(prefix, requires_grad=False):
    """The reference's call sequence (cuda_splatting.py:99-124) on the recorded arguments."""
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    view = T(prefix + "viewmatrix")
    settings = GaussianRasterizationSettings(
        image_height=int(G[prefix + "image_height"]), image_width=int(G[prefix + "image_width"]),
        tanfovx=float(G[prefix + "tanfovx"]), tanfovy=float(G[prefix + "tanfovy"]), bg=T(prefix + "bg"),
        scale_modifier=1.0, viewmatrix=view, projmatrix=T(prefix + "projmatrix"),
        sh_degree=int(G[prefix + "sh_degree"]),
        campos=torch.cat([T(prefix + "campos")[:, None], torch.zeros(3, 3, device=DEV)], 1)[:, 0],   # stride 4, as recorded
        prefiltered=False, debug=False)
    assert settings.campos.stride(0) == 4
    has_sh = (prefix + "shs") in G
    means2d = torch.zeros_like(T(prefix + "means3D"), requires_grad=True)
    img, radii = GaussianRasterizer(settings)(
        means3D=T(prefix + "means3D"), means2D=means2d, shs=T(prefix + "shs") if has_sh else None,
        colors_precomp=None if has_sh else T(prefix + "colors_precomp"), opacities=T(prefix + "opacities"),
        cov3D_precomp=T(prefix + "cov3D_precomp"))
    return img, radii


def _oracle_args(prefix):
    has_sh = (prefix + "shs") in G
    t = lambda k: torch.from_numpy(np.ascontiguousarray(G[prefix + k]))
    return dict(means=t("means3D"), cov6=t("cov3D_precomp"), opac=t("opacities")[:, 0].contiguous(),
                sh=t("shs") if has_sh else None, colors=None if has_sh else t("colors_precomp"),
                vm=t("viewmatrix").reshape(16), pm=t("projmatrix").reshape(16), campos=t("campos"),
                tanfovx=float(G[prefix + "tanfovx"]), tanfovy=float(G[prefix + "tanfovy"]),
                sh_degree=int(G[prefix + "sh_degree"]))


def _close(a, b, frac=0.995, what=""):
    a, b = np.asarray(a), np.asarray(b)
    d = np.abs(a - b)
    scale = max(1.0, float(np.abs(b).max()))
    assert (d <= 2e-5 * scale).mean() >= frac, (what, float((d <= 2e-5 * scale).mean()), float(d.max()))
    assert d.max() <= 2e-2 * scale, (what, float(d.max()))


@pytest.mark.parametrize("tag,scale_invariant", [("render_cuda", True), ("render_cuda_noscale", False)])
def test_recorded_reference_arguments_render_like_render_cuda(tag, scale_invariant):
    from pixelsplat_b200.decoder import render_cuda
    s = _scene()
    ours = render_cuda(s["extrinsics"], s["intrinsics"], s["near"], s["far"], (H, W), s["background"], s["means"],
                       s["covariances"], s["harmonics"], s["opacities"], scale_invariant=scale_invariant)
    assert ours.shape == (2, 3, H, W)
    for i in range(2):
        p = f"{tag}_{i}_"
        img, radii = _dropin(p)
        bg = tuple(float(x) for x in G[p + "bg"])
        f = util.oracle_forward(_oracle_args(p), bg, W, H)
        # the recorded arguments through the drop-in == the oracle on the same arguments (same matrices: exact decisions)
        assert np.array_equal(radii.cpu().numpy(), f.pre.radii)
        _close(img.detach().cpu().numpy(), f.color, 0.999, "drop-in vs oracle")
        assert util.psnr(img.detach().cpu().numpy(), f.color) > 60.0
        # ... == the product's batched render_cuda on the scene (matrices built on the device)
        _close(ours[i].cpu().numpy(), img.detach().cpu().numpy(), 0.995, "render_cuda vs drop-in")
        assert util.psnr(ours[i].cpu().numpy(), img.detach().cpu().numpy()) > 55.0
    assert float(ours.abs().sum()) > 0


def test_camera_setup_reproduces_the_references_matrices():
    from pixelsplat_b200.decoder.cuda_splatting import camera_setup
    s = _scene()
    for tag, scale_invariant in (("render_cuda", True), ("render_cuda_noscale", False)):
        cams = camera_setup(s["extrinsics"], s["intrinsics"], s["near"], s["far"], scale_invariant)
        for i in range(2):
            p = f"{tag}_{i}_"
            vm, pm = G[p + "viewmatrix"].reshape(16), G[p + "projmatrix"].reshape(16)
            assert np.abs(cams["viewmatrix"][i].cpu().numpy() - vm).max() <= 2e-6 * np.abs(vm).max()
            assert np.abs(cams["projmatrix"][i].cpu().numpy() - pm).max() <= 2e-6 * np.abs(pm).max()
            assert np.allclose(cams["campos"][i].cpu().numpy(), G[p + "campos"], rtol=1e-6, atol=1e-7)
            tf = cams["tanfov"][i].cpu().numpy()
            assert abs(tf[0] - float(G[p + "tanfovx"])) <= 1e-6 * tf[0] and abs(tf[1] - float(G[p + "tanfovy"])) <= 1e-6 * tf[1]
            want_scale = 1.0 / float(G["scene_near"][i]) if scale_invariant else 1.0
            assert abs(float(cams["scene_scale"][i]) - want_scale) <= 1e-6 * want_scale
            # the fused rescale: means * scene_scale is what the reference passed as means3D
            got = (s["means"][i] * cams["scene_scale"][i]).cpu().numpy()
            assert np.allclose(got, G[p + "means3D"], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("mode", ["depth", "disparity", "relative_disparity", "log"])
def test_recorded_depth_arguments_render_like_render_depth_cuda(mode):
    from pixelsplat_b200.decoder import render_depth_cuda
    s = _scene()
    ours = render_depth_cuda(s["extrinsics"], s["intrinsics"], s["near"], s["far"], (H, W), s["means"],
                             s["covariances"], s["opacities"], mode=mode)
    assert ours.shape == (2, H, W)
    for i in range(2):
        p = f"render_depth_{mode}_{i}_"
        img, _ = _dropin(p)
        ref = img.detach().mean(0).cpu().numpy()                    # cuda_splatting.py:269
        f = util.oracle_forward(_oracle_args(p), (0.0, 0.0, 0.0), W, H)
        _close(ref, f.color.mean(0), 0.999, "drop-in vs oracle")
        _close(ours[i].cpu().numpy(), ref, 0.995, mode)


def test_recorded_orthographic_arguments_render_like_render_cuda_orthographic():
    """Row a6 against values: the reference's moved-back narrow camera, our torch restatement of it, and the
    oracle -- all three on the same Gaussians."""
    from pixelsplat_b200.decoder import render_cuda_orthographic
    s = _scene(1)
    dump = {}
    ours = render_cuda_orthographic(T("ortho_extrinsics"), T("ortho_width"), T("ortho_height"), T("ortho_near"),
                                    T("ortho_far"), (H, W), s["background"][1:], s["means"], s["covariances"],
                                    s["harmonics"], s["opacities"], dump=dump)
    assert ours.shape == (1, 3, H, W)
    for k in ("extrinsics", "fov_x", "fov_y", "near", "far"):
        assert np.allclose(dump[k].cpu().numpy(), G[f"ortho_dump_{k}"], rtol=1e-5, atol=1e-6), k
    p = "render_ortho_0_"
    img, radii = _dropin(p)
    bg = tuple(float(x) for x in G[p + "bg"])
    f = util.oracle_forward(_oracle_args(p), bg, W, H)
    assert int((f.pre.radii > 0).sum()) > 50, "the orthographic view should see the scene"
    assert np.array_equal(radii.cpu().numpy(), f.pre.radii)
    _close(img.detach().cpu().numpy(), f.color, 0.999, "drop-in vs oracle")
    # the far-away camera (distance ~ 1146) amplifies float32 differences in the matrices: image-level bar
    assert util.psnr(ours[0].cpu().numpy(), img.detach().cpu().numpy()) > 40.0
    _close(ours[0].cpu().numpy(), img.detach().cpu().numpy(), 0.95, "render_cuda_orthographic vs drop-in")

"""CPU tests against tests/golden/render_cuda_args.npz: the arguments the REFERENCE's own host code
(/root/reference/src/model/decoder/cuda_splatting.py:47-269, run unmodified on a recording rasterizer
stand-in by oracle/make_render_args_golden.py) hands to `diff_gaussian_rasterization`.

They pin to the reference everything of rows a1 / a2 / a5 / a6 / b1 that does not need the missing CUDA
dependency: the boundary facts (layouts, strides, flags), `get_projection_matrix`, the depth "colours",
and -- most importantly -- the oracle's restatement of that host code (`raster_torch.prepare_view`), which
every rasterizer parity test uses to build its arguments.
"""
from pathlib import Path

import numpy as np
import torch

from oracle import raster_torch as rt
from tests import golden_util as gu

GOLD = Path(__file__).resolve().parent / "golden"
G = gu.load_npz_refs(GOLD / "render_cuda_args.npz", GOLD / "render_cuda_scene.npz")
T = lambda k: torch.from_numpy(np.asarray(G[k]))


def _scene():
    return {k: T(f"scene_{k}") for k in ("extrinsics", "intrinsics", "near", "far", "means", "covariances",
                                          "harmonics", "opacities", "background")}


def test_boundary_facts_the_reference_relies_on():
    """SURVEY.md 8 row a3 / b1, now read off the reference's own calls instead of recalled."""
    assert int(G["render_cuda_n"]) == 2 and int(G["render_ortho_n"]) == 1
    for i in range(2):
        p = f"render_cuda_{i}_"
        P = G[p + "means3D"].shape[0]
        assert G[p + "shs"].shape == (P, 25, 3) and G[p + "cov3D_precomp"].shape == (P, 6)
        assert G[p + "opacities"].shape == (P, 1) and G[p + "means2D"].shape == (P, 3)
        assert not G[p + "means2D"].any() and bool(G[p + "means2D_requires_grad"])
        assert G[p + "viewmatrix"].shape == (4, 4) and G[p + "projmatrix"].shape == (4, 4)
        assert int(G[p + "campos_stride"]) == 4 and not bool(G[p + "campos_contiguous"])     # a column of [4, 4]
        assert bool(G[p + "viewmatrix_contiguous"])              # einops materialises the "b i j -> b j i" transpose
        assert int(G[p + "sh_degree"]) == 4 and float(G[p + "scale_modifier"]) == 1.0
        assert not bool(G[p + "prefiltered"]) and not bool(G[p + "debug"])
        assert not bool(G[p + "has_scales"]) and not bool(G[p + "has_rotations"])
        assert (int(G[p + "image_height"]), int(G[p + "image_width"])) == (24, 40)
        assert "render_depth_depth_%d_shs" % i not in G
        assert G["render_depth_depth_%d_colors_precomp" % i].shape == (P, 3)
    # column-major: the recorded viewmatrix is the TRANSPOSE of inverse(extrinsics) (translation in the last row)
    s = _scene()
    ext = s["extrinsics"][1].clone()
    ext[:3, 3] *= 1 / s["near"][1]
    assert np.allclose(G["render_cuda_1_viewmatrix"], torch.linalg.inv(ext).T.numpy(), atol=1e-6)
    assert np.allclose(G["render_cuda_1_viewmatrix"][:3, 3], 0)


def test_oracle_prepare_view_reproduces_the_references_arguments():
    """`raster_torch.prepare_view` (what tests/util.view_args feeds both the C oracle and the CUDA path) against
    the reference's render_cuda: identical op sequence in float32 on the CPU -> equal to the last bit for the
    Gaussian tensors, within a few ulp for the matrices (batched vs single `inverse()` / matmul kernels)."""
    s = _scene()
    for tag, scale_invariant in (("render_cuda", True), ("render_cuda_noscale", False)):
        for i in range(2):
            a = rt.prepare_view(s["means"][0], s["covariances"][0], s["harmonics"][0], s["opacities"][0],
                                s["extrinsics"][i], s["intrinsics"][i], s["near"][i], s["far"][i],
                                dtype=torch.float32, scale_invariant=scale_invariant)
            p = f"{tag}_{i}_"
            assert np.array_equal(a["means"].numpy(), G[p + "means3D"])
            assert np.array_equal(a["cov6"].numpy(), G[p + "cov3D_precomp"])
            assert np.array_equal(a["sh"].numpy(), G[p + "shs"])
            assert np.array_equal(a["opac"].numpy(), G[p + "opacities"][:, 0])
            assert a["sh_degree"] == int(G[p + "sh_degree"])
            assert np.allclose(a["vm"].numpy(), G[p + "viewmatrix"].reshape(16), rtol=0, atol=2e-6)
            assert np.allclose(a["pm"].numpy(), G[p + "projmatrix"].reshape(16), rtol=2e-6, atol=2e-6)
            assert np.allclose(a["campos"].numpy(), G[p + "campos"], rtol=1e-7, atol=0)
            assert abs(a["tanfovx"] - float(G[p + "tanfovx"])) <= 2e-7 * float(G[p + "tanfovx"])
            assert abs(a["tanfovy"] - float(G[p + "tanfovy"])) <= 2e-7 * float(G[p + "tanfovy"])
    # use_sh = False: colours come from coefficient 0 of each channel (cuda_splatting.py:121)
    a = rt.prepare_view(s["means"][0], s["covariances"][0], T("render_depth_depth_0_colors_precomp")[:, :, None],
                        s["opacities"][0], s["extrinsics"][0], s["intrinsics"][0], s["near"][0], s["far"][0],
                        use_sh=False)
    assert a["sh"] is None and np.array_equal(a["colors"].numpy(), G["render_depth_depth_0_colors_precomp"])


def test_get_projection_matrix_matches_the_reference():
    from pixelsplat_b200.decoder import get_projection_matrix
    s = _scene()
    fov = T("proj_fov")
    got = get_projection_matrix(s["near"], s["far"], fov[:, 0], fov[:, 1])
    assert np.array_equal(got.numpy(), G["proj_matrix"])
    ref64 = rt.get_projection_matrix(float(s["near"][0]), float(s["far"][0]), float((0.5 * fov[0, 0]).tan()),
                                     float((0.5 * fov[0, 1]).tan()))
    assert np.allclose(ref64.numpy(), G["proj_matrix"][0], rtol=1e-6, atol=1e-7)


def test_depth_colours_match_the_reference():
    """render_depth_cuda's fake colours (cuda_splatting.py:238-251), all four modes."""
    from pixelsplat_b200.decoder.cuda_splatting import depth_colors
    s = _scene()
    for mode in ("depth", "disparity", "relative_disparity", "log"):
        got = depth_colors(s["extrinsics"][:, None], s["means"].expand(2, -1, -1), s["near"][:, None],
                           s["far"][:, None], mode)
        for i in range(2):
            ref = G[f"render_depth_{mode}_{i}_colors_precomp"]
            assert np.array_equal(ref[:, 0], ref[:, 1]) and np.array_equal(ref[:, 0], ref[:, 2])
            assert np.allclose(got[i, 0].numpy(), ref[:, 0], rtol=2e-6, atol=1e-6), mode
            assert not G[f"render_depth_{mode}_{i}_bg"].any()


def test_orthographic_camera_matches_the_reference():
    """render_cuda_orthographic's moved-back narrow camera (cuda_splatting.py:153-181): the dump dict and the
    matrices it hands to the rasterizer, rebuilt with the product's torch code on the CPU."""
    from pixelsplat_b200.decoder import get_projection_matrix
    ext, width, height = T("ortho_extrinsics"), T("ortho_width"), T("ortho_height")
    near, far = T("ortho_near"), T("ortho_far")
    fov_x = torch.tensor(0.1).deg2rad()
    tan_x = (0.5 * fov_x).tan()
    dist = (0.5 * width) / tan_x
    tan_y = 0.5 * height / dist
    fov_y = (2 * tan_y).atan()
    move_back = torch.eye(4).repeat(1, 1, 1)
    move_back[:, 2, 3] = -dist
    ext2 = ext @ move_back
    assert np.allclose(ext2.numpy(), G["ortho_dump_extrinsics"], rtol=1e-6)
    assert np.allclose((near + dist).numpy(), G["ortho_dump_near"]) and np.allclose((far + dist).numpy(), G["ortho_dump_far"])
    assert np.allclose(fov_y.numpy(), G["ortho_dump_fov_y"], rtol=1e-6)
    view = ext2.inverse().transpose(1, 2)
    full = view @ get_projection_matrix(near + dist, far + dist, fov_x.expand(1), fov_y).transpose(1, 2)
    scale = np.abs(G["render_ortho_0_projmatrix"]).max()
    assert np.allclose(view[0].numpy(), G["render_ortho_0_viewmatrix"], rtol=1e-5, atol=1e-3)
    assert np.abs(full[0].numpy() - G["render_ortho_0_projmatrix"]).max() <= 1e-5 * scale
    assert abs(float(tan_x) - float(G["render_ortho_0_tanfovx"])) < 1e-9
    assert abs(float(tan_y[0]) - float(G["render_ortho_0_tanfovy"])) < 1e-9

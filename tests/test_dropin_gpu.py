"""The drop-in boundary (SURVEY.md §8b): this repo's `dropin/` packages against the reference's own code path on the
same seeded inputs — its Python wrapper files (gaussian_renderer/r3dg_rasterization.py, bvh/__init__.py) over its own
pybind modules (rasterize_points.cu / bvh.cu glue + its kernels, built for sm_100).  What the reference computed is
stored in tests/golden/refparity_dropin.npz (tests/golden/make_golden_refparity.py): sha256 of the arrays compared
bit-exactly, a fixed sample and the full L2 norm of the others.  Outputs and gradients must agree to the north_star
tolerances.  Also: the full visibility bake (own tree + in-kernel sampling + own trace) against the reference's bake
(its tree + PyTorch sampling + its trace), and the sampling kernel against the reference's own
`fibonacci_sphere_sampling`."""
import os
import sys

import numpy as np
import pytest
import torch

from helpers import (GOLDEN, ROOT, GoldenCase, assert_close_to_summary, assert_visibility_close, case_inputs, digest,
                     npy, spread)

pytestmark = pytest.mark.gpu
REF_DROPIN = os.path.join(GOLDEN, "refparity_dropin.npz")
WRAPPER_IMAGES = ("color", "opacity", "depth", "feature", "normal", "surface_xyz")
RAYTRACER_P = 30_000
SAMPLING_N = (24, 32, 384)


def dropin(name):
    """The drop-in package `name` (r3dg_rasterization / bvh_tracing) as a caller that put dropin/ on its path sees it."""
    import importlib
    path = os.path.join(ROOT, "dropin")
    if path not in sys.path:
        sys.path.insert(0, path)
    return importlib.import_module(name)


def wrapper_case(P, W, H, S):
    sc, cam = case_inputs(P, W, H, S, view=4, center_shift=True)
    g = torch.Generator().manual_seed(3)
    return sc, cam, torch.tensor([0.3, 0.1, 0.7]), [torch.randn(c, H, W, generator=g) for c in (3, 1, 1, S)]


def sampling_normals():
    g = torch.Generator().manual_seed(1)
    nrm = torch.nn.functional.normalize(torch.randn(50_000, 3, generator=g), dim=-1).cuda()
    nrm[0] = torch.tensor([0.0, 0.0, -1.0]); nrm[1] = torch.tensor([0.0, 0.0, 1.0])      # the -I fallback and the identity
    return nrm


def _render_through_wrapper(mod, sc, cam, S, bg, cots):
    d = lambda t: t.cuda()
    leaves = [d(t).requires_grad_(True) for t in (sc.means3D, sc.opacities, sc.shs, sc.scales, sc.rotations, sc.features)]
    xyz, opac, shs, scales, rots, feats = leaves
    rs = mod.GaussianRasterizationSettings(
        image_height=cam.image_height, image_width=cam.image_width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, cx=cam.cx, cy=cam.cy,
        bg=d(bg), scale_modifier=1.0, viewmatrix=d(cam.viewmatrix), projmatrix=d(cam.projmatrix), sh_degree=3, campos=d(cam.campos),
        prefiltered=False, backward_geometry=True, computer_pseudo_normal=True, debug=False)
    means2D = torch.zeros_like(xyz, requires_grad=True)
    rast = mod.GaussianRasterizer(rs)
    out = rast(means3D=xyz, means2D=means2D, shs=shs, colors_precomp=None, opacities=opac, scales=scales, rotations=rots,
               cov3D_precomp=None, features=feats)
    (num_rendered, num_contrib, color, opacity, depth, feature, normal, surface_xyz, weights, radii) = out
    # the reference returns num_contrib as a NON-OWNING from_blob view of imgBuffer (rasterize_points.cu:136-139): it dangles
    # once autograd frees the saved buffers, so it is copied before backward
    num_contrib = num_contrib.clone()
    loss = sum((o * d(c)).sum() for o, c in zip((color, opacity, depth, feature), cots))
    loss.backward()
    torch.cuda.synchronize()
    vis = rast.markVisible(xyz)
    res = dict(num_rendered=int(num_rendered), num_contrib=num_contrib, color=color, opacity=opacity, depth=depth, feature=feature,
               normal=normal, surface_xyz=surface_xyz, weights=weights, radii=radii, visible=vis)
    grads = dict(means3D=xyz.grad, opacity=opac.grad, shs=shs.grad, scales=scales.grad, rotations=rots.grad, features=feats.grad,
                 means2D=means2D.grad)
    return res, grads


@pytest.mark.parametrize("P,W,H,S", [(60_000, 400, 304, 16), (300_000, 800, 800, 5)], ids=["60k-S16", "300k-S5"])
def test_dropin_wrapper_matches_reference_stock_path(P, W, H, S):
    mod = dropin("r3dg_rasterization")
    assert "relightable3dgaussian_b200" in mod._C.__file__
    g = GoldenCase(REF_DROPIN, f"wrapper_{P}_{W}x{H}_S{S}")
    sc, cam, bg, cots = wrapper_case(P, W, H, S)
    oo, og = _render_through_wrapper(mod, sc, cam, S, bg, cots)
    assert oo["num_rendered"] == int(g["num_rendered"])
    for n in ("radii", "num_contrib", "visible"):
        assert digest(oo[n]) == str(g[n]), n
    for n in WRAPPER_IMAGES:
        assert_close_to_summary(g, n, oo[n], max_abs=1e-4)
    vis = np.nonzero(npy(oo["radii"]) > 0)[0]
    for n in og:
        assert og[n] is not None, n
        assert_close_to_summary(g, "grad_" + n, og[n], rows=vis, rel=1e-3)


def _bvh_scene(P):
    sc, _ = case_inputs(P, 64, 64, 0)
    d = lambda t: t.cuda()
    return d(sc.means3D), d(sc.scales), d(sc.rotations), d(sc.opacities[:, 0].contiguous()), d(sc.normals)


def test_dropin_raytracer_matches_reference_raytracer():
    from oracle import oracle_sampling
    mod = dropin("bvh_tracing")
    g = GoldenCase(REF_DROPIN, "raytracer")
    xyz, s, r, op, nrm = _bvh_scene(RAYTRACER_P)
    icov = oracle_sampling.inverse_covariance(s, r)
    a = mod.RayTracer(xyz, s, r)
    assert digest(a.tree) == str(g["tree"]) and digest(a.morton) == str(g["morton"])   # topology + Morton codes bit-exact
    dirs, _ = oracle_sampling.sample_incident_rays(nrm, False, 24)
    va = a.trace_visibility(xyz[:, None].expand_as(dirs), dirs, xyz, icov, op, nrm)
    assert_visibility_close(g, "vis", va["visibility"], max_flips=1e-3, max_abs=1e-4)


def test_sampling_kernel_vs_reference_function():
    """r3dg_sample_incident_dirs vs the reference's own fibonacci_sphere_sampling (utils/graphics_utils.py:9-37) run on
    a B200, deterministic and random-rotate variants."""
    from relightable3dgaussian_b200 import raytracer
    g = GoldenCase(REF_DROPIN, "sampling")
    nrm = sampling_normals()
    for N in SAMPLING_N:
        d, a = raytracer.sample_incident_rays(nrm, False, N)
        assert tuple(d.shape) == tuple(g[f"dirs_{N}_shape"]) and tuple(a.shape) == tuple(g[f"areas_{N}_shape"])
        assert digest(npy(a).view(np.int32)) == str(g[f"areas_{N}"])
        assert np.abs(spread(d, k=4096) - g[f"dirs_{N}"]).max() <= 5e-7, N                   # unit vectors: a few ulp at most
    # random rotation: same phase numbers through both
    torch.manual_seed(5)
    d, _ = raytracer.fibonacci_sphere_sampling(nrm, 32, random_rotate=True)
    assert np.abs(spread(d, k=4096) - g["dirs_rot"]).max() <= 5e-6


@pytest.mark.parametrize("P,N", [(100_000, 32), (40_000, 64)])
def test_full_bake_parity_own_tree_vs_reference_tree(P, N):
    """update_visibility end to end: OUR tree (exact refit) + in-kernel sampling + our trace, against the REFERENCE's
    bake (its racy-refit tree, PyTorch sampling, its trace kernel, its chunk loop).  Visibility is a step function of T
    at 0.9, so the flip rate across that cliff is the meaningful figure (north_star)."""
    from oracle import oracle_sampling
    from relightable3dgaussian_b200 import raytracer
    g = GoldenCase(REF_DROPIN, f"bake_{P}_{N}")
    xyz, s, r, op, nrm = _bvh_scene(P)
    icov = oracle_sampling.inverse_covariance(s, r)
    assert (raytracer.inverse_covariance(s, r) - icov).abs().max().item() <= 1e-3 * icov.abs().max().item()
    vis, dirs, areas = raytracer.update_visibility(xyz, s, r, icov, op, nrm, N)
    assert tuple(vis.shape) == tuple(g["vis_shape"]) == (P, N, 1) and dirs.shape == (P, N, 3)
    assert digest(npy(areas).view(np.int32)) == str(g["areas"])
    assert np.abs(spread(dirs, k=4096) - g["dirs"]).max() <= 5e-7
    flip, err = assert_visibility_close(g, "vis", vis, max_flips=1e-3, max_abs=1e-4)
    print(f"[bake] P={P} N={N}: flip rate {flip:.2e} (every 8th Gaussian), max-abs on agreeing sampled rays {err:.2e}")

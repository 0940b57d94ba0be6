"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the C ABI of
libr3dg_b200.so via the reference-shaped host API; the CPU oracle and outputs of the unmodified
reference CUDA kernels stored under tests/golden/ are the checkers.

Tolerances (BASELINE.json north_star): images <= 1e-4 max-abs, gradients <= 1e-3 relative,
tile / sort indices bit-exact."""
import glob
import os
import sys

import numpy as np
import pytest
import torch

from helpers import (GOLDEN, ROOT, GoldenCase, assert_close_to_summary, case_inputs, digest, max_rel_above_floor, npy,
                     oracle_kwargs, rel_l2)

pytestmark = pytest.mark.gpu
RASTER_CASES = sorted(glob.glob(os.path.join(GOLDEN, "raster_*.npz")))
GRADS = ["dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dfeatures", "dL_dcov3D", "dL_dsh",
         "dL_dscales", "dL_drotations"]


@pytest.fixture(scope="module")
def C():
    from relightable3dgaussian_b200 import _C_raster
    assert torch.cuda.is_available()
    return _C_raster


def dev(t):
    return torch.Tensor([]) if t is None else torch.as_tensor(t).cuda()


def run_ours(C, *, means3D, opacities, viewmatrix, projmatrix, campos, bg, W, H, tan_fovx, tan_fovy, cx, cy,
             shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None, features=None,
             sh_degree=3, pseudo=True, cots=None, backward_geometry=True):
    P = means3D.shape[0]
    feats = dev(features) if features is not None else torch.empty((P, 0), device="cuda")
    a = dict(bg=dev(bg), means3D=dev(means3D), feats=feats, colors=dev(colors_precomp), opac=dev(opacities),
             scales=dev(scales), rots=dev(rotations), cov=dev(cov3D_precomp), view=dev(viewmatrix),
             proj=dev(projmatrix), sh=dev(shs), campos=dev(campos))
    out = C.rasterize_gaussians(a["bg"], a["means3D"], a["feats"], a["colors"], a["opac"], a["scales"], a["rots"], 1.0,
                                a["cov"], a["view"], a["proj"], tan_fovx, tan_fovy, cx, cy, H, W, a["sh"], sh_degree,
                                a["campos"], False, pseudo, False)
    names = ["num_rendered", "n_contrib", "color", "opacity", "depth", "feature", "normal", "surface_xyz", "weights",
             "radii", "geom", "binning", "img"]
    o = dict(zip(names, out))
    S = feats.shape[1]
    o["mid"] = lambda n: C.debug_intermediate(n, P, S, W, H, o["geom"], o["img"], o["binning"], o["num_rendered"])
    if cots is not None:
        g = C.rasterize_gaussians_backward(a["bg"], a["means3D"], a["feats"], o["radii"], a["colors"], a["scales"],
                                           a["rots"], 1.0, a["cov"], a["view"], a["proj"], tan_fovx, tan_fovy,
                                           dev(cots[0]), dev(cots[1]), dev(cots[2]), dev(cots[3]), a["sh"], sh_degree,
                                           a["campos"], o["geom"], o["num_rendered"], o["binning"], o["img"],
                                           backward_geometry, False)
        o["grads"] = dict(zip(GRADS, g))
    torch.cuda.synchronize()
    return o


def golden_kwargs(g):
    P, W, H, S, view, deg, R = [int(x) for x in g["meta"]]
    tfx, tfy, cx, cy = [float(x) for x in g["tanfov"]]
    kw = dict(means3D=g["in_means3D"], opacities=g["in_opacities"], viewmatrix=g["in_viewmatrix"],
              projmatrix=g["in_projmatrix"], campos=g["in_campos"], bg=g["in_bg"], W=W, H=H, tan_fovx=tfx, tan_fovy=tfy,
              cx=cx, cy=cy, features=g["in_features"] if S else None, sh_degree=deg)
    if str(g["mode"]) == "sh_sr":
        kw.update(shs=g["in_shs"], scales=g["in_scales"], rotations=g["in_rotations"])
    else:
        kw.update(colors_precomp=g["in_colors_precomp"], cov3D_precomp=g["in_cov3D_precomp"])
    return kw, (P, W, H, S, R)


@pytest.mark.parametrize("path", RASTER_CASES, ids=[os.path.basename(p)[7:-4] for p in RASTER_CASES])
def test_matches_reference_cuda_golden(C, path):
    g = np.load(path)
    kw, (P, W, H, S, R) = golden_kwargs(g)
    o = run_ours(C, cots=[g["cot_color"], g["cot_opacity"], g["cot_depth"], g["cot_feature"]], **kw)
    vis = g["out_radii"] > 0
    assert o["num_rendered"] == R
    assert np.array_equal(npy(o["radii"]), g["out_radii"])                          # bit-exact indices
    assert np.array_equal(npy(o["mid"]("tiles_touched")), g["mid_tiles_touched"])
    assert np.array_equal(npy(o["mid"]("point_list_keys")), g["mid_point_list_keys"])
    assert np.array_equal(npy(o["mid"]("point_list")), g["mid_point_list"])
    T = ((W + 15) // 16) * ((H + 15) // 16)
    assert np.array_equal(npy(o["mid"]("ranges")), g["mid_ranges"][:T])
    assert np.array_equal(npy(o["n_contrib"]).reshape(-1), g["mid_n_contrib"])
    for n in ("depths", "means2D", "conic_opacity"):
        assert np.array_equal(npy(o["mid"](n))[vis].view(np.uint32), g["mid_" + n][vis].view(np.uint32)), n
    for n in ("color", "opacity", "depth", "feature", "normal", "surface_xyz"):       # <= 1e-4 (in fact bit-equal)
        if g["out_" + n].size:
            assert np.abs(npy(o[n]) - g["out_" + n]).max() <= 1e-6, n
    assert np.abs(npy(o["weights"]) - g["out_weights"]).max() < 1e-4
    names = [n for n in GRADS if g["grad_" + n].size and np.abs(g["grad_" + n]).max() > 0]
    for n in names:
        assert rel_l2(npy(o["grads"][n]), g["grad_" + n]) < 1e-3, n
        assert max_rel_above_floor(npy(o["grads"][n]), g["grad_" + n], floor=1e-3) < 1e-2, n


def test_binning_multi_window_path(C, monkeypatch):
    """bin_scatter stages a chunk's instances in shared memory; a chunk that does not fit is handled in
    several windows of tiles.  Force a tiny staging area and require the same bit-exact lists."""
    g = np.load(RASTER_CASES[0])
    kw, (P, W, H, S, R) = golden_kwargs(g)
    monkeypatch.setenv("R3DG_BIN_STAGE_CAP", "1")          # clamped up to the chunk length by the library
    o = run_ours(C, **kw)
    assert o["num_rendered"] == R
    assert np.array_equal(npy(o["mid"]("point_list")), g["mid_point_list"])
    T = ((W + 15) // 16) * ((H + 15) // 16)
    assert np.array_equal(npy(o["mid"]("ranges")), g["mid_ranges"][:T])
    assert np.array_equal(npy(o["n_contrib"]).reshape(-1), g["mid_n_contrib"])


def _forward_vs_oracle(C, P, W, H, boost):
    from oracle import oracle
    sc, cam = case_inputs(P, W, H, 0, view=1, scale_boost=boost)
    kw = oracle_kwargs(sc, cam, torch.tensor([0.1, 0.0, 0.3]))
    extra = dict(shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations))
    o = run_ours(C, pseudo=False, **kw, **extra)
    f = oracle.rasterize_forward(computer_pseudo_normal=False, **kw, **extra)
    assert o["num_rendered"] == f["binned"]["num_rendered"] > P
    assert np.array_equal(npy(o["mid"]("point_list")).view(np.uint32), f["binned"]["point_list"])
    assert np.array_equal(npy(o["mid"]("ranges")).view(np.uint32), f["binned"]["ranges"])
    # the CPU oracle's expf differs from CUDA's in the last ulp: a pair whose alpha sits exactly on the 1/255
    # threshold can flip (2 of 8.3M pixels at 4K, 3.5e-3 each); against the reference CUDA kernels the images are
    # bit-identical (golden tests)
    d = np.abs(npy(o["color"]) - f["img"]["color"]).max(axis=0)
    assert (d > 1e-4).mean() < 1e-5 and d.max() < 1e-2


@pytest.mark.parametrize("W,H,P,boost", [(1920, 1080, 20_000, 1.0), (3840, 2160, 6_000, 1.0), (50, 1200, 3_000, 2.0)],
                         ids=["1080p", "4k", "tall"])
def test_binning_many_tiles(C, W, H, P, boost):
    """8160 / 32400 tiles and a 4 x 75 tile strip: the per-tile tables of the binning kernels scale with the tile
    count and the staging area shrinks accordingly (multi-window scatter at 4K)."""
    _forward_vs_oracle(C, P, W, H, boost)


def test_binning_long_chunks(C, monkeypatch):
    """More Gaussians than 2048 x (rows of the chunk x tile matrix): chunks grow beyond 2048 Gaussians
    (P > 2M at the default 1024 rows).  Emulated by shrinking the matrix to 3 rows."""
    monkeypatch.setenv("R3DG_BIN_MAX_CHUNKS", "3")
    _forward_vs_oracle(C, 20_000, 320, 232, 1.5)


@pytest.mark.parametrize("S,pseudo", [(0, False), (5, True), (16, True)])
def test_matches_cpu_oracle_midsize(C, S, pseudo):
    from oracle import oracle
    sc, cam = case_inputs(20_000, 320, 232, S, view=3, scale_boost=1.5)
    bg = torch.tensor([0.2, 0.4, 0.1])
    kw = oracle_kwargs(sc, cam, bg)
    extra = dict(shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations),
                 features=npy(sc.features) if S else None)
    rng = np.random.default_rng(5)
    cots = [rng.standard_normal((c, 232, 320)).astype(np.float32) for c in (3, 1, 1, S)]
    o = run_ours(C, cots=cots, pseudo=pseudo, **kw, **extra)
    f = oracle.rasterize_forward(computer_pseudo_normal=pseudo, **kw, **extra)
    bk = {k: v for k, v in {**kw, **extra}.items() if k not in ("opacities", "cx", "cy")}
    gr = oracle.rasterize_backward(f, dL_dcolor=cots[0], dL_dopacity=cots[1], dL_ddepth=cots[2], dL_dfeature=cots[3], **bk)
    assert o["num_rendered"] == f["binned"]["num_rendered"]
    assert np.array_equal(npy(o["radii"]), f["pre"]["radii"])
    assert np.array_equal(npy(o["mid"]("point_list")).view(np.uint32), f["binned"]["point_list"])
    assert np.array_equal(npy(o["mid"]("ranges")).view(np.uint32), f["binned"]["ranges"])
    assert (npy(o["n_contrib"]).reshape(-1) != f["img"]["n_contrib"]).mean() < 1e-3
    for n in ("color", "opacity", "depth", "feature"):
        if f["img"][n].size:
            assert np.abs(npy(o[n]) - f["img"][n]).max() <= 1e-4, n
    if pseudo:
        assert np.quantile(np.abs(npy(o["normal"]) - f["normal"]).max(axis=0), 0.99) < 1e-3
        assert np.abs(npy(o["surface_xyz"]) - f["surface_xyz"]).max() < 1e-2
    else:
        assert not npy(o["normal"]).any() and not npy(o["surface_xyz"]).any()
    for n in GRADS:
        if gr[n].size:
            assert rel_l2(npy(o["grads"][n]), gr[n]) < 1e-3, n


REF_PARITY = os.path.join(GOLDEN, "refparity_raster.npz")
PARITY_INDICES = ("radii", "tiles_touched", "point_list", "point_list_keys", "ranges", "n_contrib")
PARITY_IMAGES = ("color", "opacity", "depth", "feature", "normal", "surface_xyz")


def parity_inputs(P, W, H, S, view, center_shift, backward=True, recipe="shell-v1", sh_degree=3, M=16, scale_boost=1.0):
    """One seeded comparison with the unmodified reference kernels: (case key, rasterizer kwargs, cotangents or None)."""
    sc, cam = case_inputs(P, W, H, S, view=view, center_shift=center_shift, recipe=recipe, scale_boost=scale_boost)
    kw = oracle_kwargs(sc, cam, torch.tensor([0.0, 0.5, 1.0]))
    kw.update(shs=np.ascontiguousarray(npy(sc.shs)[:, :M]), scales=npy(sc.scales), rotations=npy(sc.rotations),
              features=npy(sc.features) if S else None, sh_degree=sh_degree)
    g = torch.Generator().manual_seed(2)
    cots = [torch.randn(c, H, W, generator=g) for c in (3, 1, 1, S)] if backward else None
    key = f"{recipe}_{P}_{W}x{H}_S{S}_v{view}{'c' if center_shift else ''}_deg{sh_degree}M{M}_b{scale_boost:g}{'' if backward else '_fwd'}"
    return key, kw, cots


def parity_outputs(o, grads, W, H):
    """The arrays a comparison with the reference looks at, from a forward dict (intermediates through o["mid"]) and
    the gradient dict (None: forward only)."""
    T = ((W + 15) // 16) * ((H + 15) // 16)
    out = {n: o["mid"](n) for n in ("tiles_touched", "point_list", "point_list_keys")}
    out.update(radii=o["radii"], ranges=o["mid"]("ranges")[:T], n_contrib=o["n_contrib"].reshape(-1), weights=o["weights"],
               **{n: o[n] for n in PARITY_IMAGES}, **{"grad_" + n: t for n, t in (grads or {}).items()})
    return out


def _reference_parity(C, *case, **kwcase):
    """Our kernels vs the UNMODIFIED reference kernels on the same inputs (tests/golden/refparity_raster.npz, made by
    make_golden_refparity.py): tile / sort indices bit-exact (sha256 of the whole arrays), images <= 1e-4 max-abs,
    all nine gradients <= 1e-3 relative (north_star), on a fixed sample of each array plus its full L2 norm."""
    key, kw, cots = parity_inputs(*case, **kwcase)
    g = GoldenCase(REF_PARITY, key)
    o = run_ours(C, cots=cots, **kw)
    got = parity_outputs(o, o.get("grads"), kw["W"], kw["H"])
    assert o["num_rendered"] == int(g["num_rendered"])
    for n in PARITY_INDICES:
        assert digest(got[n]) == str(g[n]), n
    vis = np.nonzero(npy(o["radii"]) > 0)[0]
    for n in PARITY_IMAGES:
        if n in g:
            assert_close_to_summary(g, n, got[n], max_abs=1e-4)
    assert_close_to_summary(g, "weights", got["weights"], rows=vis, max_abs=1e-3 * max(1.0, float(g["weights_maxabs"])))
    for n in GRADS:
        if "grad_" + n in g:
            assert_close_to_summary(g, "grad_" + n, got["grad_" + n], rows=vis, rel=1e-3)
    assert (cots is not None) == any("grad_" + n in g for n in GRADS)


def test_matches_live_reference_kernels_if_built(C):
    _reference_parity(C, 200_000, 640, 480, 5, view=5, center_shift=True)


@pytest.mark.parametrize("P,W,H,S,view,shift,bwd", [
    (300_000, 800, 800, 0, 1, False, False),        # BASELINE config #2: forward raster only
    (300_000, 800, 800, 0, 2, False, True),         # BASELINE config #3: full fwd+bwd training step shape
    (1_000_000, 800, 800, 5, 0, False, True),       # the headline bench configuration, exactly
    (1_500_000, 1600, 1200, 16, 3, True, True),     # BASELINE config #4 raster shape: S = 16, off-centre principal point
    (2_000_000, 1920, 1080, 16, 6, False, True),    # BASELINE config #5 raster shape
], ids=["cfg2-300k-fwd", "cfg3-300k-fwdbwd", "headline-1M-S5", "cfg4-1.5M-1600x1200-S16", "cfg5-2M-1080p-S16"])
def test_live_reference_parity_at_benchmark_sizes(C, P, W, H, S, view, shift, bwd):
    _reference_parity(C, P, W, H, S, view, shift, backward=bwd)


@pytest.mark.parametrize("S", [1, 3, 7, 9, 12, 13, 17, 20, 21, 24, 28, 33])
def test_every_channel_group_instantiation(C, S):
    """The compositors are templates on the number of 4-channel groups (S = 0..33 forward, 0..24 backward, the
    reference's limits forward.cu:312 / backward.cu:449): every instantiation against the reference kernels."""
    _reference_parity(C, 6_000, 208, 144, S, view=S % 8, center_shift=bool(S & 1), backward=S <= 24, scale_boost=2.0)


@pytest.mark.parametrize("deg,M", [(0, 1), (1, 4), (2, 9), (3, 16), (1, 16), (0, 16)])
def test_sh_degrees_and_row_widths(C, deg, M):
    """SH rows of 12 / 48 / 108 / 192 bytes: the bulk-copy slab path needs 16-byte rows, the others take the
    transposed LDGSTS path (projection.cu); degrees below the stored width ignore the upper coefficients."""
    _reference_parity(C, 9_000, 200, 136, 5, view=deg + 2, center_shift=False, sh_degree=deg, M=M, scale_boost=1.5)


def test_backward_launch_order_follows_measured_forward_work(C):
    """The forward compositor records, per half-tile CTA, how many entries its busiest warp composited; the backward's
    CTAs are launched in that order (coarse 64-bucket LPT).  Invariants against n_contrib, and the order is a permutation."""
    P, W, H, S = 40_000, 400, 304, 5
    sc, cam = case_inputs(P, W, H, S, view=2, scale_boost=1.5)
    kw = oracle_kwargs(sc, cam, torch.tensor([0.0, 0.0, 0.0]))
    g = torch.Generator().manual_seed(3)
    cots = [torch.randn(c, H, W, generator=g) for c in (3, 1, 1, S)]
    o = run_ours(C, cots=cots, shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations), features=npy(sc.features), **kw)
    gx, gy = (W + 15) // 16, (H + 15) // 16
    work = o["mid"]("bwd_work").long()                      # [T, 2]: rows 0-7 / 8-15 of the tile
    order = o["mid"]("bwd_order").long()
    nc = torch.zeros(gy * 16, gx * 16, dtype=torch.int64, device="cuda")
    nc[:H, :W] = o["n_contrib"].long()
    half_max = nc.view(gy, 2, 8, gx, 16).amax(dim=(2, 4)).permute(0, 2, 1).reshape(gy * gx, 2)   # deepest contributor per half tile
    assert bool(((work > 0) == (half_max > 0)).all())
    assert bool((work <= half_max).all())                   # composited entries are a subset of the positions walked
    assert torch.equal(torch.sort(order).values, torch.arange(2 * gx * gy, device="cuda"))
    keys = work.reshape(-1)[order]
    shift = max(int(keys.max()).bit_length() - 6, 0)
    assert bool(((keys[:-1] >> shift) >= (keys[1:] >> shift)).all())


def test_full_size_properties(C):
    """BASELINE.json headline size (1M Gaussians, 800x800): size-independent properties."""
    P, W, H, S = 1_000_000, 800, 800, 5
    sc, cam = case_inputs(P, W, H, S, view=0)
    bg = torch.tensor([0.1, 0.2, 0.3])
    kw = oracle_kwargs(sc, cam, bg)
    extra = dict(shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations), features=npy(sc.features))
    g = torch.Generator().manual_seed(4)
    cots = [torch.randn(c, H, W, generator=g) for c in (3, 1, 1, S)]
    o = run_ours(C, cots=cots, **kw, **extra)
    R = o["num_rendered"]
    keys, pl, ranges, tiles = o["mid"]("point_list_keys"), o["mid"]("point_list"), o["mid"]("ranges"), o["mid"]("tiles_touched")
    assert R == int(tiles.long().sum()) and keys.numel() == R
    assert bool((keys[1:] >= keys[:-1]).all())                                    # sortedness
    same = keys[1:] == keys[:-1]
    assert bool((pl[1:][same] > pl[:-1][same]).all())                             # stability (tie order)
    lens = (ranges[:, 1].long() - ranges[:, 0].long())
    assert int(lens.sum()) == R and bool((lens >= 0).all())
    assert torch.equal(torch.bincount(keys >> 32, minlength=ranges.shape[0]), lens)  # ranges partition the list
    assert torch.equal(torch.bincount(pl.long(), minlength=P), tiles.long())          # each Gaussian once per touched tile
    depths = o["mid"]("depths")
    assert torch.equal((keys & 0xFFFFFFFF).int(), depths.view(torch.int32)[pl.long()])
    assert bool(torch.isfinite(o["color"]).all()) and float(o["opacity"].min()) >= 0 and float(o["opacity"].max()) <= 1 + 1e-5
    tile_of_pix = (torch.arange(H, device="cuda")[:, None] // 16) * 50 + torch.arange(W, device="cuda")[None, :] // 16
    assert bool((o["n_contrib"].long() <= lens[tile_of_pix]).all())
    # determinism of the forward (idempotence) and linearity of the backward in the cotangents
    o2 = run_ours(C, cots=[2 * c for c in cots], **kw, **extra)
    for n in ("color", "depth", "feature", "normal", "n_contrib", "radii"):
        assert torch.equal(o[n], o2[n]), n
    for n in ("dL_dmeans3D", "dL_dsh", "dL_dscales", "dL_dopacity"):
        assert rel_l2(npy(o2["grads"][n]), 2 * npy(o["grads"][n])) < 1e-4, n
    # total opacity-weight checksum: sum_p weights[p] == sum_pixels opacity (same quantity, two reductions)
    assert abs(float(o["weights"].double().sum()) - float(o["opacity"].double().sum())) / float(o["opacity"].double().sum()) < 1e-4


def test_edge_cases(C):
    from oracle import oracle
    cam = case_inputs(4, 100, 60, 0)[1]
    base = dict(viewmatrix=npy(cam.viewmatrix), projmatrix=npy(cam.projmatrix), campos=npy(cam.campos),
                bg=np.array([0.5, 0.25, 1.0], np.float32), W=100, H=60, tan_fovx=cam.tanfovx, tan_fovy=cam.tanfovy,
                cx=cam.cx, cy=cam.cy)
    z = lambda *s: np.zeros(s, np.float32)
    # P == 0: background image, zero instances
    o = run_ours(C, means3D=z(0, 3), opacities=z(0, 1), shs=z(0, 16, 3), scales=z(0, 3), rotations=z(0, 4), **base)
    assert o["num_rendered"] == 0 and np.allclose(npy(o["color"])[2], 1.0) and not npy(o["n_contrib"]).any()
    # all Gaussians behind the camera
    sc, _ = case_inputs(300, 100, 60, 5)
    behind = npy(sc.means3D + cam.campos * 3.0)
    rng = np.random.default_rng(0)
    cots = [rng.standard_normal((c, 60, 100)).astype(np.float32) for c in (3, 1, 1, 5)]
    o = run_ours(C, means3D=behind, opacities=npy(sc.opacities), shs=npy(sc.shs), scales=npy(sc.scales),
                 rotations=npy(sc.rotations), features=npy(sc.features), cots=cots, **base)
    assert o["num_rendered"] == 0 and not npy(o["radii"]).any()
    assert all(not npy(v).any() for v in o["grads"].values())                      # every grad row written as zero
    assert not npy(C.mark_visible(dev(behind), dev(base["viewmatrix"]), dev(base["projmatrix"]))).any()
    # one huge Gaussian covering the whole screen (radius >> image) + ragged image size
    big = dict(means3D=z(1, 3), opacities=np.full((1, 1), 0.9, np.float32), shs=z(1, 16, 3),
               scales=np.full((1, 3), 2.0, np.float32), rotations=np.array([[1, 0, 0, 0]], np.float32))
    o = run_ours(C, **big, **base)
    f = oracle.rasterize_forward(**big, **base)
    assert o["num_rendered"] == f["binned"]["num_rendered"] == 7 * 4
    assert np.abs(npy(o["color"]) - f["img"]["color"]).max() < 1e-5
    # S = 33 (forward maximum, forward.cu:312) forward-only; S = 24 backward maximum; S = 25 backward refuses
    sc, _ = case_inputs(500, 100, 60, 33, scale_boost=4.0)
    kw = dict(means3D=npy(sc.means3D), opacities=npy(sc.opacities), shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations))
    o = run_ours(C, features=npy(sc.features), **kw, **base)
    f = oracle.rasterize_forward(features=npy(sc.features), **kw, **base)
    assert np.abs(npy(o["feature"]) - f["img"]["feature"]).max() < 1e-4
    cots24 = [rng.standard_normal((c, 60, 100)).astype(np.float32) for c in (3, 1, 1, 24)]
    o = run_ours(C, features=npy(sc.features[:, :24]), cots=cots24, **kw, **base)
    f = oracle.rasterize_forward(features=npy(sc.features[:, :24]), **kw, **base)
    gr = oracle.rasterize_backward(f, dL_dcolor=cots24[0], dL_dopacity=cots24[1], dL_ddepth=cots24[2], dL_dfeature=cots24[3],
                                   features=npy(sc.features[:, :24]), **{k: v for k, v in kw.items() if k != "opacities"},
                                   **{k: v for k, v in base.items() if k not in ("cx", "cy")})
    for n in ("dL_dfeatures", "dL_dmeans3D", "dL_dsh"):
        assert rel_l2(npy(o["grads"][n]), gr[n]) < 1e-3, n
    cots25 = [rng.standard_normal((c, 60, 100)).astype(np.float32) for c in (3, 1, 1, 25)]
    with pytest.raises(RuntimeError):
        run_ours(C, features=npy(sc.features[:, :25]), cots=cots25, **kw, **base)
    # speculative binning capacity too small -> transparent rerun with identical results
    from relightable3dgaussian_b200 import _C_raster
    ref_out = run_ours(C, features=npy(sc.features[:, :5]), **kw, **base)
    for st in _C_raster._state.values():
        st["capacity"] = 0
    sc2, _ = case_inputs(500, 100, 60, 5, scale_boost=12.0)       # > 4 instances per Gaussian on average
    kw2 = dict(means3D=npy(sc2.means3D), opacities=npy(sc2.opacities), shs=npy(sc2.shs), scales=npy(sc2.scales), rotations=npy(sc2.rotations))
    o = run_ours(C, features=npy(sc2.features), **kw2, **base)
    f = oracle.rasterize_forward(features=npy(sc2.features), **kw2, **base)
    assert o["num_rendered"] == f["binned"]["num_rendered"] > 4 * 500 + 4096 or o["num_rendered"] == f["binned"]["num_rendered"]
    assert np.array_equal(npy(o["mid"]("point_list")).view(np.uint32), f["binned"]["point_list"])
    assert ref_out["num_rendered"] > 0


def test_operator_surface_and_autograd(C):
    from relightable3dgaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    from oracle import oracle
    sc, cam = case_inputs(5000, 208, 144, 5, view=4, scale_boost=2.0)
    bg = torch.tensor([0.3, 0.3, 0.3])
    rs = GaussianRasterizationSettings(144, 208, cam.tanfovx, cam.tanfovy, cam.cx, cam.cy, bg.cuda(), 1.0,
                                       cam.viewmatrix.cuda(), cam.projmatrix.cuda(), 3, cam.campos.cuda(), False, True, True, False)
    assert GaussianRasterizationSettings._fields == ("image_height", "image_width", "tanfovx", "tanfovy", "cx", "cy", "bg",
                                                     "scale_modifier", "viewmatrix", "projmatrix", "sh_degree", "campos",
                                                     "prefiltered", "backward_geometry", "computer_pseudo_normal", "debug")
    rast = GaussianRasterizer(rs)
    leaf = lambda t: t.cuda().requires_grad_(True)
    m3, op, sh, s, r, ft = map(leaf, (sc.means3D, sc.opacities, sc.shs, sc.scales, sc.rotations, sc.features))
    m2 = torch.zeros_like(m3, requires_grad=True)
    with pytest.raises(Exception):
        rast(means3D=m3, means2D=m2, opacities=op, scales=s, rotations=r)                       # neither shs nor colours
    with pytest.raises(Exception):
        rast(means3D=m3, means2D=m2, opacities=op, shs=sh, scales=s, rotations=r, cov3D_precomp=torch.zeros(5000, 6).cuda())
    out = rast(means3D=m3, means2D=m2, opacities=op, shs=sh, scales=s, rotations=r, features=ft)
    assert len(out) == 10 and isinstance(out[0], int) and out[1].dtype == torch.int32 and out[9].dtype == torch.int32
    g = torch.Generator().manual_seed(0)
    cots = [torch.randn(c, 144, 208, generator=g) for c in (3, 1, 1, 5)]
    loss = sum((o * c.cuda()).sum() for o, c in zip(out[2:6], cots)) + out[6].sum() + out[8].sum()   # normal/weights grads are ignored
    loss.backward()
    kw = oracle_kwargs(sc, cam, bg)
    ex = dict(shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations), features=npy(sc.features))
    f = oracle.rasterize_forward(**kw, **ex)
    gr = oracle.rasterize_backward(f, dL_dcolor=npy(cots[0]), dL_dopacity=npy(cots[1]), dL_ddepth=npy(cots[2]), dL_dfeature=npy(cots[3]),
                                   **{k: v for k, v in {**kw, **ex}.items() if k not in ("opacities", "cx", "cy")})
    for t, n in ((m3, "dL_dmeans3D"), (m2, "dL_dmeans2D"), (op, "dL_dopacity"), (sh, "dL_dsh"), (s, "dL_dscales"),
                 (r, "dL_drotations"), (ft, "dL_dfeatures")):
        assert t.grad is not None and rel_l2(npy(t.grad), gr[n]) < 1e-3, n
    vis = rast.markVisible(m3.detach())
    assert vis.dtype == torch.bool and bool(vis.all())
    # backward_geometry=False drops the feature term from dL/dalpha (backward.cu:563-566)
    rs2 = rs._replace(backward_geometry=False)
    for t in (m3, m2, op, sh, s, r, ft):
        t.grad = None
    out2 = GaussianRasterizer(rs2)(means3D=m3, means2D=m2, opacities=op, shs=sh, scales=s, rotations=r, features=ft)
    (out2[5] * cots[3].cuda()).sum().backward()
    gr2 = oracle.rasterize_backward(f, dL_dcolor=np.zeros_like(npy(cots[0])), dL_dopacity=np.zeros_like(npy(cots[1])),
                                    dL_ddepth=np.zeros_like(npy(cots[2])), dL_dfeature=npy(cots[3]), backward_geometry=False,
                                    **{k: v for k, v in {**kw, **ex}.items() if k not in ("opacities", "cx", "cy")})
    assert rel_l2(npy(ft.grad), gr2["dL_dfeatures"]) < 1e-3
    assert float(op.grad.abs().max()) == 0.0 and float(np.abs(gr2["dL_dopacity"]).max()) == 0.0


def test_dropin_module_names():
    sys.path.insert(0, os.path.join(ROOT, "dropin"))
    import importlib
    mod = importlib.import_module("r3dg_rasterization")
    for n in ("rasterize_gaussians", "rasterize_gaussians_backward", "mark_visible"):
        assert callable(getattr(mod._C, n))
    assert hasattr(mod, "GaussianRasterizer") and hasattr(mod, "GaussianRasterizationSettings")


def test_deferred_count_option(C):
    """Opt-in host run-ahead: same results, `num_rendered` resolves lazily (tests/test_feature_ops_gpu.py covers
    the overflow repair); the first _LEARN forwards of a shape and undifferentiated forwards stay synchronous."""
    from relightable3dgaussian_b200 import rasterizer, _C_raster
    from relightable3dgaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    sc, cam = case_inputs(4000, 160, 96, 5, view=2, scale_boost=3.0)
    rs = GaussianRasterizationSettings(96, 160, cam.tanfovx, cam.tanfovy, cam.cx, cam.cy, torch.zeros(3).cuda(), 1.0,
                                       cam.viewmatrix.cuda(), cam.projmatrix.cuda(), 3, cam.campos.cuda(), False, True, True, False)
    def run():
        leaf = lambda t: t.cuda().requires_grad_(True)
        m3, op, sh, s, r, ft = map(leaf, (sc.means3D, sc.opacities, sc.shs, sc.scales, sc.rotations, sc.features))
        out = GaussianRasterizer(rs)(means3D=m3, means2D=torch.zeros_like(m3, requires_grad=True), opacities=op, shs=sh,
                                     scales=s, rotations=r, features=ft)
        (out[2].sum() + out[5].sum()).backward()
        return out, sh.grad
    _C_raster._state.clear()
    ref_out, ref_g = run()
    rasterizer.set_deferred_count(True)
    try:
        for i in range(_C_raster._LEARN - 1):
            out, g = run()
            assert isinstance(out[0], int)                      # still learning the counts of this shape: synchronous
        out, g = run()
        assert isinstance(out[0], _C_raster.DeferredCount) and int(out[0]) == ref_out[0] and not out[0].overflowed
        assert torch.equal(out[2], ref_out[2]) and torch.equal(out[1], ref_out[1])
        assert rel_l2(npy(g), npy(ref_g)) < 1e-5
        sc2, _ = case_inputs(300, 160, 96, 5, view=2, scale_boost=40.0)
        leaf = lambda t: t.cuda()
        big = lambda: GaussianRasterizer(rs)(means3D=leaf(sc2.means3D), means2D=torch.zeros(300, 3).cuda(), opacities=leaf(sc2.opacities),
                                             shs=leaf(sc2.shs), scales=leaf(sc2.scales), rotations=leaf(sc2.rotations), features=leaf(sc2.features))
        out = big()                                             # new shape, nothing requires grad: synchronous, retried on a miss
        assert isinstance(out[0], int) and out[0] > 4 * 300 + 4096
    finally:
        rasterizer.set_deferred_count(False)


def test_bulk_copy_record_staging_variant_is_bit_identical(C):
    """r3dg_tune("composite_bulk", 1): the forward compositor stages its records with per-lane TMA bulk copies
    (cp.async.bulk + mbarrier) instead of the register prefetch — same arithmetic, so identical images and counters."""
    from relightable3dgaussian_b200 import _lib
    for path in RASTER_CASES[:2]:
        g = np.load(path)
        kw, (P, W, H, S, R) = golden_kwargs(g)
        a = run_ours(C, **kw)
        prev = _lib.tune("composite_bulk", 1)
        try:
            b = run_ours(C, **kw)
        finally:
            _lib.tune("composite_bulk", prev)
        for n in ("color", "opacity", "depth", "feature", "n_contrib", "normal"):
            assert torch.equal(a[n], b[n]), n
        # weights are accumulated with float atomics, so two runs differ in the last bits of the larger values
        assert bool(((a["weights"] - b["weights"]).abs() < 1e-5 * b["weights"].abs().clamp_min(1.0)).all())
    sc, cam = case_inputs(300_000, 800, 800, 16, view=1)
    kw = oracle_kwargs(sc, cam, torch.tensor([0.0, 0.5, 1.0]))
    extra = dict(shs=npy(sc.shs), scales=npy(sc.scales), rotations=npy(sc.rotations), features=npy(sc.features))
    a = run_ours(C, **kw, **extra)
    prev = _lib.tune("composite_bulk", 1)
    try:
        b = run_ours(C, **kw, **extra)
    finally:
        _lib.tune("composite_bulk", prev)
    for n in ("color", "feature", "n_contrib"):
        assert torch.equal(a[n], b[n]), n

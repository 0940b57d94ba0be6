"""GPU parity of the BVH visibility path (through the C ABI): LBVH topology / Morton codes / boxes
bit-exact, visibility <= 1e-4 with the flip rate across the T < 0.9 cliff reported and bounded."""
import glob
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, GoldenCase, assert_visibility_close, bvh_case, digest, inverse_covariance, npy

pytestmark = pytest.mark.gpu
CASES = sorted(glob.glob(os.path.join(GOLDEN, "bvh_*.npz")))


def build_ours(means3D, scales, rotations):
    from relightable3dgaussian_b200.raytracer import RayTracer
    rt = RayTracer(means3D.cuda(), scales.cuda(), rotations.cuda())
    torch.cuda.synchronize()
    return rt


def check_tree(rt, ref_nodes, ref_aabbs, ref_morton, exact_aabbs=None):
    """nodes / morton bit-exact.  Boxes: the leaf half bit-exact; the internal half must equal the
    exact bottom-up min/max (CPU oracle) when given.  The reference's own refit (construct.cu:229-265)
    reads child boxes without a fence after the flag CAS, so on a large GPU some of ITS internal
    boxes are stale (too small, never too large): they must be contained in ours."""
    P = rt.morton.shape[0]
    assert np.array_equal(npy(rt.morton).view(np.uint64), np.asarray(ref_morton).view(np.uint64))
    assert np.array_equal(npy(rt.tree), ref_nodes)
    ours = npy(rt.aabb)
    assert np.array_equal(ours[P - 1:].view(np.uint32), ref_aabbs[P - 1:].view(np.uint32))
    assert (ours[:P - 1, :3] <= ref_aabbs[:P - 1, :3]).all() and (ours[:P - 1, 3:] >= ref_aabbs[:P - 1, 3:]).all()
    if exact_aabbs is not None:
        assert np.array_equal(ours.view(np.uint32), exact_aabbs.view(np.uint32))
    return float((ours[:P - 1] != ref_aabbs[:P - 1]).any(axis=1).mean())


def compare_vis(vis, cont, ref_vis, ref_cont):
    flips = ((vis == 0) != (ref_vis == 0)).mean()
    same = (vis == 0) == (ref_vis == 0)
    return flips, (np.abs(vis - ref_vis)[same].max() if same.any() else 0.0), (cont != ref_cont)[same].mean()


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[4:-4] for p in CASES])
def test_matches_reference_bvh_golden(path):
    from relightable3dgaussian_b200 import _C_bvh
    g = np.load(path)
    t = lambda k: torch.from_numpy(g["in_" + k])
    from oracle import oracle
    rt = build_ours(t("means3D"), t("scales"), t("rotations"))
    exact = oracle.bvh_build(g["in_means3D"], g["in_scales"], g["in_rotations"])[1]
    check_tree(rt, g["nodes"], g["aabbs"], g["morton"], exact)
    # trace OUR kernel on the REFERENCE's tree (its own boxes) so the traversal is the same
    cont, vis = _C_bvh.trace_bvh_opacity(torch.from_numpy(g["nodes"]).cuda(), torch.from_numpy(g["aabbs"]).cuda(),
                                         t("rays_o").cuda(), t("rays_d").cuda(), t("means3D").cuda(),
                                         t("inv_cov").cuda(), t("opacity").cuda(), t("normals").cuda())
    torch.cuda.synchronize()
    assert vis.shape == g["visibility"].shape and cont.dtype == torch.int32
    flips, err, cdiff = compare_vis(npy(vis), npy(cont), g["visibility"], g["contribute"])
    assert flips <= 2e-3 and err <= 1e-4 and cdiff <= 2e-3, (flips, err, cdiff)
    v = npy(vis)
    assert ((v == 0) | (v >= 0.9)).all()


def test_matches_cpu_oracle_and_live_reference():
    from oracle import oracle
    c = bvh_case("cube-v1", 20_000, 600, 48, 2.0, seed=5)
    d = {k: v.cuda() for k, v in c.items()}
    rt = build_ours(c["means3D"], c["scales"], c["rotations"])
    nodes, aabbs, morton = oracle.bvh_build(npy(c["means3D"]), npy(c["scales"]), npy(c["rotations"]))
    check_tree(rt, nodes, aabbs, morton, aabbs)
    # host mirror: un-expanded origins + fused 0.05 offset == reference call with materialised rays
    n_src, N = 600, 48
    res = rt.trace_visibility(d["means3D"][:n_src, None].expand(n_src, N, 3), d["rays_d"], d["means3D"], d["inv_cov"],
                              d["opacity"], d["normals"])
    vis, cont = npy(res["visibility"])[..., 0], npy(res["contribute"])[..., 0]
    oc, ov = oracle.bvh_trace_opacity(nodes, aabbs, npy(c["rays_o"]), npy(c["rays_d"]), npy(c["means3D"]), npy(c["inv_cov"]),
                                      npy(c["opacity"]), npy(c["normals"]))
    flips, err, cdiff = compare_vis(vis, cont, ov, oc)
    assert flips <= 2e-3 and err <= 1e-4 and cdiff <= 5e-3, (flips, err, cdiff)
    assert 0.02 < (ov == 0).mean() < 0.98                                     # the case exercises both outcomes
    # the reference's own tree and trace (tests/golden/refparity_bvh.npz, make_golden_refparity.py); its boxes are stored
    # as the internal ones that differ from the exact refit, so its tree is rebuilt here bit for bit
    g = GoldenCase(os.path.join(GOLDEN, "refparity_bvh.npz"), "bvh_cube_20000")
    ref_aabbs = aabbs.copy()
    ref_aabbs[g["stale_rows"].astype(np.int64)] = g["stale_aabbs"]
    assert digest(ref_aabbs.view(np.int32)) == str(g["aabbs"])
    stale = check_tree(rt, nodes, ref_aabbs, morton)
    assert digest(nodes) == str(g["nodes"]) and digest(np.asarray(morton).view(np.int64)) == str(g["morton"])
    print(f"reference internal boxes that differ from the exact refit (its missing-fence race): {stale:.4%}")
    # same tree (the reference's) for both tracers
    from relightable3dgaussian_b200 import _C_bvh
    _, ov2 = _C_bvh.trace_bvh_opacity(rt.tree, torch.from_numpy(ref_aabbs).cuda(), d["rays_o"], d["rays_d"], d["means3D"],
                                      d["inv_cov"], d["opacity"], d["normals"])
    flips, err = assert_visibility_close(g, "vis", ov2, max_flips=1e-3, max_abs=1e-4, step=1)
    print(f"trace vs reference: flip rate {flips:.2e}, max-abs on agreeing sampled rays {err:.2e}")


def test_update_visibility_shapes_and_edge_cases():
    from relightable3dgaussian_b200.raytracer import RayTracer, update_visibility
    from relightable3dgaussian_b200 import _C_bvh
    c = bvh_case("shell-v1", 3000, 8, 8, 3.0)
    d = {k: v.cuda() for k, v in c.items()}
    vis, dirs, areas = update_visibility(d["means3D"], d["scales"], d["rotations"], d["inv_cov"], d["opacity"], d["normals"], 40)
    assert vis.shape == (3000, 40, 1) and dirs.shape == (3000, 40, 3) and areas.shape == (3000, 40, 1)
    assert torch.allclose(areas, torch.full_like(areas, 2 * np.pi)) and ((vis == 0) | (vis >= 0.9)).all()
    # P == 2 (smallest tree with an internal node) and zero rays
    rt = RayTracer(d["means3D"][:2], d["scales"][:2], d["rotations"][:2])
    assert rt.tree.shape == (3, 5) and int(rt.tree[0, 4]) == 2 and sorted(rt.tree[0, 1:3].tolist()) == [1, 2]
    cont, opa = _C_bvh.trace_bvh_opacity(rt.tree, rt.aabb, torch.zeros(0, 3).cuda(), torch.zeros(0, 3).cuda(), d["means3D"][:2],
                                         d["inv_cov"][:2], d["opacity"][:2], d["normals"][:2])
    assert cont.shape == (0,) and opa.shape == (0,)
    with pytest.raises(NotImplementedError):
        _C_bvh.trace_bvh(rt.tree, rt.aabb, None, None, None, None, None)
    # axis-aligned rays (zero direction components -> IEEE inf/NaN slab arithmetic, utility.cuh:37-64)
    o = d["means3D"][:64] + torch.tensor([0.0, 0.0, 2.5]).cuda()
    dd = torch.tensor([0.0, 0.0, -1.0]).cuda().expand(64, 3).contiguous()
    rt = RayTracer(d["means3D"], d["scales"], d["rotations"])
    from oracle import oracle
    nodes, aabbs, _ = oracle.bvh_build(npy(c["means3D"]), npy(c["scales"]), npy(c["rotations"]))
    cont, opa = _C_bvh.trace_bvh_opacity(rt.tree, rt.aabb, o.contiguous(), dd, d["means3D"], d["inv_cov"], d["opacity"], d["normals"])
    oc, ov = oracle.bvh_trace_opacity(nodes, aabbs, npy(o), npy(dd), npy(c["means3D"]), npy(c["inv_cov"]), npy(c["opacity"]), npy(c["normals"]))
    assert ((npy(opa) == 0) != (ov == 0)).mean() <= 0.05


def test_sampling_kernel_matches_reference_golden():
    """r3dg_sample_incident_dirs vs tests/golden/sampling.npz (outputs of the reference's own functions)."""
    from relightable3dgaussian_b200 import raytracer
    g = np.load(os.path.join(GOLDEN, "sampling.npz"))
    n = torch.from_numpy(g["normals"]).cuda()
    for N in (24, 32, 100):
        d, a = raytracer.sample_incident_rays(n, False, N)
        assert d.shape == (257, N, 3) and np.array_equal(npy(a), g[f"areas_{N}"])
        assert np.abs(npy(d) - g[f"dirs_{N}"]).max() <= 5e-7, N          # CPU libm vs CUDA sinf/cosf: <= a few ulp of a unit vector
        assert np.abs(np.linalg.norm(npy(d), axis=-1) - 1).max() < 1e-6
    # batched normals keep their leading shape (graphics_utils.py:11-13,32-35)
    d, a = raytracer.sample_incident_rays(n[:256].reshape(16, 16, 3), False, 24)
    assert d.shape == (16, 16, 24, 3) and a.shape == (16, 16, 24, 1)
    assert np.abs(npy(d).reshape(256, 24, 3) - g["dirs_24"][:256]).max() <= 5e-7


def test_bake_kernel_equals_sampler_plus_trace_and_cpu_oracle():
    """r3dg_bvh_bake_visibility (directions generated in the trace kernel, Morton-ordered rays) must equal the two-step
    path it fuses (r3dg_sample_incident_dirs -> trace_visibility) ray for ray, and the CPU oracle's trace on the same
    tree up to the T < 0.9 cliff; partial slot ranges touch only their own Gaussians' rows."""
    from oracle import oracle
    from relightable3dgaussian_b200 import raytracer
    c = bvh_case("cube-v1", 6000, 8, 8, 2.0, seed=3)
    d = {k: v.cuda() for k, v in c.items()}
    N = 40
    rt = build_ours(c["means3D"], c["scales"], c["rotations"])
    full = rt.bake_visibility(d["means3D"], d["inv_cov"], d["opacity"], d["normals"], N, want_contribute=True)
    dirs, areas = raytracer.sample_incident_rays(d["normals"], False, N)
    assert torch.equal(full["incident_dirs"], dirs) and torch.equal(full["incident_areas"], areas)
    two = rt.trace_visibility(d["means3D"][:, None].expand_as(dirs), dirs, d["means3D"], d["inv_cov"], d["opacity"], d["normals"])
    assert torch.equal(full["visibility"], two["visibility"]) and torch.equal(full["contribute"], two["contribute"])
    nodes, aabbs, _ = oracle.bvh_build(npy(c["means3D"]), npy(c["scales"]), npy(c["rotations"]))
    ro = npy(d["means3D"][:, None] + dirs * 0.05).reshape(-1, 3)
    oc, ov = oracle.bvh_trace_opacity(nodes, aabbs, ro, npy(dirs).reshape(-1, 3), npy(c["means3D"]), npy(c["inv_cov"]),
                                      npy(c["opacity"]), npy(c["normals"]))
    flips, err, _ = compare_vis(npy(full["visibility"]).reshape(-1), npy(full["contribute"]).reshape(-1), ov, oc)
    assert flips <= 2e-3 and err <= 1e-4, (flips, err)
    # slots [1000, 3500): exactly those Gaussians' rows, nothing else
    part = rt.bake_visibility(d["means3D"], d["inv_cov"], d["opacity"], d["normals"], N, first_slot=1000, count=2500)
    P = 6000
    objs = rt.tree[P - 1 + 1000:P - 1 + 3500, 3].long()
    mask = torch.zeros(P, dtype=torch.bool, device="cuda"); mask[objs] = True
    assert torch.equal(part["visibility"][mask], full["visibility"][mask]) and not part["visibility"][~mask].any()
    assert not part["incident_dirs"][~mask].any() and torch.equal(part["incident_dirs"][mask], dirs[mask])

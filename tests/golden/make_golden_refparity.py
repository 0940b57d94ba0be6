#!/usr/bin/env python3
"""Generates tests/golden/refparity_*.npz on a GPU from the UNMODIFIED reference CUDA code built into oracle/_ref
(oracle/build_ref.sh: its kernels behind the raw-pointer shims; oracle/build_ref_ext.sh: its own pybind modules and
Python wrappers).  For every case of the reference comparisons in test_raster_gpu.py, test_dropin_gpu.py and
test_bvh_gpu.py it runs the reference on the test's seeded inputs and keeps what the test compares against: the
sha256 of every array compared bit-exactly, and a fixed sample plus the full L2 norm of every array compared within
a tolerance (tests/helpers.py: digest / summarize / summarize_visibility).

    python tests/golden/make_golden_refparity.py <outdir>
"""
import importlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [TESTS, ROOT]
from helpers import bvh_case, digest, npy, pack_golden_case, spread, summarize, summarize_visibility  # noqa: E402
from oracle import oracle, oracle_sampling, ref_gpu  # noqa: E402
import test_dropin_gpu as tdrop  # noqa: E402
import test_raster_gpu as traster  # noqa: E402

# the arguments of every _reference_parity call in test_raster_gpu.py
RASTER_CASES = (
    [((200_000, 640, 480, 5), dict(view=5, center_shift=True))] +
    [((P, W, H, S), dict(view=v, center_shift=sh, backward=b)) for P, W, H, S, v, sh, b in [
        (300_000, 800, 800, 0, 1, False, False), (300_000, 800, 800, 0, 2, False, True), (1_000_000, 800, 800, 5, 0, False, True),
        (1_500_000, 1600, 1200, 16, 3, True, True), (2_000_000, 1920, 1080, 16, 6, False, True)]] +
    [((6_000, 208, 144, S), dict(view=S % 8, center_shift=bool(S & 1), backward=S <= 24, scale_boost=2.0))
     for S in (1, 3, 7, 9, 12, 13, 17, 20, 21, 24, 28, 33)] +
    [((9_000, 200, 136, 5), dict(view=deg + 2, center_shift=False, sh_degree=deg, M=M, scale_boost=1.5))
     for deg, M in [(0, 1), (1, 4), (2, 9), (3, 16), (1, 16), (0, 16)]])
WRAPPER_CASES = [(60_000, 400, 304, 16), (300_000, 800, 800, 5)]        # test_dropin_gpu.py
BAKE_CASES = [(100_000, 32), (40_000, 64)]


def raster_record(o, grads, W, H):
    got = traster.parity_outputs(o, grads, W, H)
    rec = {"num_rendered": np.int64(o["num_rendered"])}
    rec.update({n: np.str_(digest(got[n])) for n in traster.PARITY_INDICES})
    vis = np.nonzero(npy(o["radii"]) > 0)[0]
    for n in traster.PARITY_IMAGES:
        if got[n].numel():
            rec.update(summarize(n, got[n]))
    rec.update(summarize("weights", got["weights"], rows=vis))
    for n, t in (grads or {}).items():
        if t.numel() and float(t.abs().max()) > 0:
            rec.update(summarize("grad_" + n, t, rows=vis))
    return rec


def raster():
    rec = {}
    for args, kwargs in RASTER_CASES:
        key, kw, cots = traster.parity_inputs(*args, **kwargs)
        ref = ref_gpu.RefRasterizer()
        tk = {k: (traster.dev(v) if isinstance(v, np.ndarray) else v) for k, v in kw.items() if v is not None}
        ro = ref.forward(**tk)
        grads = None
        if cots is not None:
            grads = ref.backward(ro, dL_dcolor=traster.dev(cots[0]), dL_dopacity=traster.dev(cots[1]), dL_ddepth=traster.dev(cots[2]),
                                 dL_dfeature=traster.dev(cots[3]),
                                 **{k: v for k, v in tk.items() if k in ("means3D", "viewmatrix", "projmatrix", "campos", "bg",
                                                                         "tan_fovx", "tan_fovy", "shs", "scales", "rotations", "features", "sh_degree")})
            grads = {n: grads[n] for n in traster.GRADS}
        torch.cuda.synchronize()
        o = dict(ro, n_contrib=ref.intermediate("n_contrib"), mid=ref.intermediate)
        rec.update(pack_golden_case(key, raster_record(o, grads, kw["W"], kw["H"])))
        print(f"[raster] {key}: R={ro['num_rendered']}", flush=True)
        del ref
        torch.cuda.empty_cache()
    return rec


def reference_fibonacci():
    py = os.path.join(ROOT, "oracle", "_ref", "py")
    sys.path.insert(0, py)
    try:
        return importlib.import_module("utils.graphics_utils").fibonacci_sphere_sampling
    finally:
        sys.path.remove(py)


def dropin():
    rec = {}
    theirs = ref_gpu.load_reference_wrapper("raster", "ref")
    for P, W, H, S in WRAPPER_CASES:
        sc, cam, bg, cots = tdrop.wrapper_case(P, W, H, S)
        ro, rg = tdrop._render_through_wrapper(theirs, sc, cam, S, bg, cots)
        vis = np.nonzero(npy(ro["radii"]) > 0)[0]
        r = {"num_rendered": np.int64(ro["num_rendered"]), "radii": np.str_(digest(ro["radii"])),
             "num_contrib": np.str_(digest(ro["num_contrib"])), "visible": np.str_(digest(ro["visible"]))}
        for n in tdrop.WRAPPER_IMAGES:
            r.update(summarize(n, ro[n]))
        for n, t in rg.items():
            r.update(summarize("grad_" + n, t, rows=vis))
        rec.update(pack_golden_case(f"wrapper_{P}_{W}x{H}_S{S}", r))
        print(f"[dropin] wrapper P={P}: R={ro['num_rendered']}", flush=True)
    bvh = ref_gpu.load_reference_wrapper("bvh", "ref")
    xyz, s, r_, op, nrm = tdrop._bvh_scene(tdrop.RAYTRACER_P)
    icov = oracle_sampling.inverse_covariance(s, r_)
    rt = bvh.RayTracer(xyz, s, r_)
    dirs, _ = oracle_sampling.sample_incident_rays(nrm, False, 24)
    vb = rt.trace_visibility(xyz[:, None].expand_as(dirs), dirs, xyz, icov, op, nrm)
    rec.update(pack_golden_case("raytracer", {"tree": np.str_(digest(rt.tree)), "morton": np.str_(digest(rt.morton)),
                                      **summarize_visibility("vis", vb["visibility"])}))
    fib = reference_fibonacci()
    nrm = tdrop.sampling_normals()
    r = {}
    for N in tdrop.SAMPLING_N:
        d, a = fib(nrm, N, random_rotate=False)
        r.update({f"dirs_{N}": spread(d, k=4096), f"dirs_{N}_shape": np.array(d.shape), f"areas_{N}": np.str_(digest(npy(a).view(np.int32))),
                  f"areas_{N}_shape": np.array(a.shape)})
    torch.manual_seed(5)
    r["dirs_rot"] = spread(fib(nrm, 32, random_rotate=True)[0], k=4096)
    rec.update(pack_golden_case("sampling", r))
    for P, N in BAKE_CASES:
        xyz, s, r_, op, nrm = tdrop._bvh_scene(P)
        icov = oracle_sampling.inverse_covariance(s, r_)
        rvis, rdirs, rareas, kind = ref_gpu.reference_update_visibility(xyz, s, r_, icov, op, nrm, N)
        rec.update(pack_golden_case(f"bake_{P}_{N}", {"vis_shape": np.array(rvis.shape), "dirs": spread(rdirs, k=4096),
                                              "areas": np.str_(digest(npy(rareas).view(np.int32))),
                                              **summarize_visibility("vis", rvis)}))
        print(f"[dropin] bake P={P} N={N}: {kind}", flush=True)
    return rec


def bvh_live():
    """test_bvh_gpu.py::test_matches_cpu_oracle_and_live_reference: the reference's tree and its trace on that tree.  Its
    boxes are kept as the internal ones that differ from the exact refit (CPU oracle): its refit is racy, see
    test_bvh_gpu.check_tree."""
    c = bvh_case("cube-v1", 20_000, 600, 48, 2.0, seed=5)
    d = {k: v.cuda() for k, v in c.items()}
    P = c["means3D"].shape[0]
    rn, ra, rm = ref_gpu.ref_bvh_create(d["means3D"], d["scales"], d["rotations"])
    rc, rv = ref_gpu.ref_bvh_trace_opacity(rn, ra, d["rays_o"], d["rays_d"], d["means3D"], d["inv_cov"], d["opacity"], d["normals"])
    torch.cuda.synchronize()
    ra = npy(ra)
    exact = oracle.bvh_build(npy(c["means3D"]), npy(c["scales"]), npy(c["rotations"]))[1]
    stale = np.nonzero((ra[:P - 1] != exact[:P - 1]).any(axis=1))[0]
    print(f"[bvh] reference internal boxes that differ from the exact refit: {stale.size} of {P - 1}", flush=True)
    return pack_golden_case("bvh_cube_20000", {
        "nodes": np.str_(digest(rn)), "morton": np.str_(digest(rm)), "aabbs": np.str_(digest(ra.view(np.int32))),
        "stale_rows": stale.astype(np.float64), "stale_aabbs": ra[stale], **summarize_visibility("vis", rv, step=1)})


def main(outdir):
    os.makedirs(outdir, exist_ok=True)
    assert ref_gpu.available() and ref_gpu.bvh_available() and ref_gpu.ext_available("raster") and ref_gpu.ext_available("bvh"), \
        "build oracle/_ref first (oracle/build_ref.sh, oracle/build_ref_ext.sh)"
    for name, make in (("raster", raster), ("dropin", dropin), ("bvh", bvh_live)):
        path = os.path.join(outdir, f"refparity_{name}.npz")
        np.savez_compressed(path, **make())
        print(f"wrote {path}: {os.path.getsize(path) / 1e3:.0f} kB", flush=True)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)

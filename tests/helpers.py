"""Shared test utilities: seeded cases, conversions, comparison helpers."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from relightable3dgaussian_b200 import synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def sh_case(P, seed):
    """Inputs of BASELINE.json config #1: sh [P,3,16] (channel-major, utils/sh_utils.py:77), unit dirs."""
    g = torch.Generator().manual_seed(1000 + seed)
    sh = torch.randn(P, 3, 16, generator=g) * 0.3
    dirs = torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1)
    return sh, dirs


def npy(t):
    return None if t is None else t.detach().cpu().numpy()


def case_inputs(P, W, H, S, view=1, recipe="shell-v1", seed=0, scale_boost=1.0, center_shift=False):
    sc = synth.make_scene(P, recipe, seed, S)
    if scale_boost != 1.0:
        sc = sc._replace(scales=sc.scales * scale_boost)
    cam = synth.make_camera(view, W, H, center_shift=center_shift)
    return sc, cam


def oracle_kwargs(sc, cam, bg):
    return dict(means3D=npy(sc.means3D), opacities=npy(sc.opacities), viewmatrix=npy(cam.viewmatrix),
                projmatrix=npy(cam.projmatrix), campos=npy(cam.campos), bg=npy(bg),
                W=cam.image_width, H=cam.image_height, tan_fovx=cam.tanfovx, tan_fovy=cam.tanfovy,
                cx=cam.cx, cy=cam.cy)


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


def max_rel_above_floor(a, b, floor=1e-6):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    m = np.abs(b) > floor * (np.abs(b).max() + 1e-30)
    if not m.any():
        return 0.0
    return float((np.abs(a - b)[m] / np.abs(b)[m]).max())


def digest(a):
    """sha256 of an integer / boolean array's values (as int64): stands in for a bit-exact comparison with a
    stored reference array that is too large to keep."""
    a = npy(a) if torch.is_tensor(a) else np.asarray(a)
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int64).tobytes()).hexdigest()


def spread(a, rows=None, k=128):
    """k evenly spaced elements of `a` (of its rows `rows` only, when given), flattened, as float32: a fixed
    sample that stands in for a stored reference array that is too large to keep."""
    a = npy(a) if torch.is_tensor(a) else np.asarray(a)
    a = a.reshape(a.shape[0], -1)[rows].reshape(-1) if rows is not None else a.reshape(-1)
    if a.size == 0:
        return np.zeros(0, np.float32)
    return a[np.linspace(0, a.size - 1, min(k, a.size)).astype(np.int64)].astype(np.float32)


def summarize(prefix, a, rows=None):
    """What a golden file keeps of a float array: a fixed sample (`spread`), its full L2 norm and max-abs."""
    a = np.asarray(npy(a) if torch.is_tensor(a) else a, np.float64)
    return {prefix: spread(a, rows), prefix + "_l2": np.float64(np.linalg.norm(a)),
            prefix + "_maxabs": np.float64(np.abs(a).max(initial=0.0))}


def assert_close_to_summary(g, prefix, a, rows=None, max_abs=None, rel=None):
    """`a` against a stored `summarize` record.  max_abs: every sampled element within it, and the full L2 norms
    within max_abs * sqrt(n) (what a full max-abs bound implies); rel: relative L2 error of the sample below it,
    and the full L2 norms within rel (what a full relative L2 bound implies)."""
    a = np.asarray(npy(a) if torch.is_tensor(a) else a, np.float64)
    ref = g[prefix]
    s = spread(a, rows, k=ref.size)
    assert s.shape == ref.shape, (prefix, s.shape, ref.shape)
    dn = abs(float(np.linalg.norm(a)) - float(g[prefix + "_l2"]))
    if max_abs is not None:
        assert np.abs(s - ref).max(initial=0.0) <= max_abs, (prefix, np.abs(s - ref).max())
        assert dn <= max_abs * np.sqrt(a.size), (prefix, dn)
    if rel is not None:
        assert rel_l2(s, ref) < rel, (prefix, rel_l2(s, ref))
        assert dn < rel * float(g[prefix + "_l2"]), (prefix, dn)


def summarize_visibility(prefix, vis, step=8):
    """What a golden file keeps of a visibility tensor [P, ...]: for every `step`-th Gaussian, which rays are blocked
    (bit-packed) and a fixed sample of the values."""
    v = np.asarray(npy(vis) if torch.is_tensor(vis) else vis)[::step].reshape(-1)
    return {prefix + "_blocked": np.packbits(v == 0), prefix + "_values": spread(v, k=2048)}


def assert_visibility_close(g, prefix, vis, max_flips, max_abs, step=8):
    """`vis` against a `summarize_visibility` record: the share of rays whose blocked / visible outcome differs (the
    T < 0.9 cliff) at most max_flips, the sampled values of rays on the same side within max_abs."""
    v = np.asarray(npy(vis) if torch.is_tensor(vis) else vis)[::step].reshape(-1)
    blocked = np.unpackbits(g[prefix + "_blocked"], count=v.size).astype(bool)
    flips = float((blocked != (v == 0)).mean())
    s, ref = spread(v, k=2048), g[prefix + "_values"]
    same = (s == 0) == (ref == 0)
    err = float(np.abs(s - ref)[same].max(initial=0.0))
    assert flips <= max_flips and err <= max_abs, (prefix, flips, err)
    return flips, err


_KINDS = {"float32": "f4", "uint8": "u1", "str": "U64"}


def pack_golden_case(key, rec):
    """One case of a golden file that holds several, as a few npz entries (an npz of many small arrays is mostly zip
    headers): the values of all arrays of one kind (float32, uint8, str, float64 for the rest) concatenated, and an
    index of `name kind offset shape` lines.  GoldenCase reads it back."""
    groups, index = {}, []
    for name, v in rec.items():
        v = np.asarray(v)
        kind = "str" if v.dtype.kind == "U" else v.dtype.name if v.dtype.name in _KINDS else "float64"
        arrs = groups.setdefault(kind, [])
        index.append(f"{name} {kind} {sum(a.size for a in arrs)} {','.join(map(str, v.shape))}")
        arrs.append(v.reshape(-1).astype(_KINDS.get(kind, "f8")))
    return {f"{key}.index": np.array(index), **{f"{key}.{k}": np.concatenate(a) for k, a in groups.items()}}


class GoldenCase:
    """One case of a golden file written with pack_golden_case: a mapping name -> array."""

    def __init__(self, path, key):
        z = np.load(path)
        assert f"{key}.index" in z.files, \
            f"{os.path.basename(path)} has no case {key}: regenerate it with tests/golden/make_golden_refparity.py"
        self.items = {}
        for line in z[f"{key}.index"]:
            name, kind, off, shape = str(line).split(" ")
            shape = tuple(int(x) for x in shape.split(",") if x)
            flat = z[f"{key}.{kind}"]
            self.items[name] = flat[int(off):int(off) + int(np.prod(shape))].reshape(shape)

    def __getitem__(self, name):
        return self.items[name]

    def __contains__(self, name):
        return name in self.items


def inverse_covariance(scales, rotations):
    """scene/gaussian_model.py:257-260 + utils/general_utils.py:151-160 (strip_symmetric of
    L L^T with L = R diag(1/s)); torch ops, device of the inputs."""
    r = rotations
    norm = torch.sqrt(r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1] + r[:, 2] * r[:, 2] + r[:, 3] * r[:, 3])
    q = r / norm[:, None]
    R = torch.zeros((q.size(0), 3, 3), device=r.device)
    rr, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R[:, 0, 0] = 1 - 2 * (y * y + z * z); R[:, 0, 1] = 2 * (x * y - rr * z); R[:, 0, 2] = 2 * (x * z + rr * y)
    R[:, 1, 0] = 2 * (x * y + rr * z); R[:, 1, 1] = 1 - 2 * (x * x + z * z); R[:, 1, 2] = 2 * (y * z - rr * x)
    R[:, 2, 0] = 2 * (x * z - rr * y); R[:, 2, 1] = 2 * (y * z + rr * x); R[:, 2, 2] = 1 - 2 * (x * x + y * y)
    L = torch.zeros((q.size(0), 3, 3), dtype=torch.float, device=r.device)
    inv_s = 1 / scales
    L[:, 0, 0] = inv_s[:, 0]; L[:, 1, 1] = inv_s[:, 1]; L[:, 2, 2] = inv_s[:, 2]
    L = R @ L
    cov = L @ L.transpose(1, 2)
    return torch.stack([cov[:, 0, 0], cov[:, 0, 1], cov[:, 0, 2], cov[:, 1, 1], cov[:, 1, 2], cov[:, 2, 2]], dim=-1).contiguous()


def bvh_case(recipe, P, n_src, N, boost, seed=3):
    """Seeded BVH / visibility case: P Gaussians, rays from the first n_src of them along N
    Fibonacci directions around the FLIPPED normal (so that they run through the scene),
    origins pre-offset by 0.05 d like bvh/__init__.py:63."""
    from oracle.oracle_sampling import fibonacci_sphere_sampling
    sc = synth.make_scene(P, recipe, seed, 0)
    scales = sc.scales * boost
    normals = sc.normals
    dirs, _ = fibonacci_sphere_sampling(-normals[:n_src], N, random_rotate=False)
    rays_o = (sc.means3D[:n_src, None] + dirs * 0.05).contiguous()
    return dict(means3D=sc.means3D, scales=scales.contiguous(), rotations=sc.rotations, opacity=sc.opacities[:, 0].contiguous(),
                normals=normals, inv_cov=inverse_covariance(scales, sc.rotations), rays_o=rays_o, rays_d=dirs.contiguous())


def shading_case(P, N, He, seed):
    """Seeded inputs of `rendering_equation` (neilf.py:339): activated material parameters, SH
    incident light, raw env map (softplus applied by the light object), baked visibility / dirs."""
    from oracle.oracle_sampling import fibonacci_sphere_sampling
    g = torch.Generator().manual_seed(500 + seed)
    n = torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1)
    dirs, areas = fibonacci_sphere_sampling(n, N, random_rotate=False)
    vis = torch.where(torch.rand(P, N, 1, generator=g) < 0.4, torch.zeros(P, N, 1), 0.9 + 0.1 * torch.rand(P, N, 1, generator=g))
    return dict(base_color=torch.sigmoid(torch.randn(P, 3, generator=g)) * 0.77 + 0.03,
                roughness=torch.sigmoid(torch.randn(P, 1, generator=g)) * 0.9 + 0.09,
                normals=(n + 0.05 * torch.randn(P, 3, generator=g)).contiguous(),       # deliberately not unit length
                viewdirs=torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1),
                incidents=(torch.randn(P, 16, 3, generator=g) * 0.3).contiguous(),
                env_raw=torch.randn(1, He, 2 * He, 3, generator=g),
                visibility=vis.contiguous(), incident_dirs=dirs.contiguous(), incident_areas=areas.contiguous(),
                cot_pbr=torch.randn(P, 3, generator=g), cot_diffuse=torch.randn(P, 3, generator=g),
                cot_specular=torch.randn(P, 3, generator=g))


def adam_case():
    """Seeded optimiser case shared by tests/golden/make_golden_adam.py and the tests: three parameter
    groups shaped like the reference's (xyz [P,3], f_rest [P,15,3], opacity [P,1]) with its learning
    rates (arguments/__init__.py), 7 steps of gradients (exact zeros for half of the f_rest rows: never
    seen Gaussians, eps = 1e-15 decides; an all-zero step for xyz), one lr edit at step 5."""
    g = torch.Generator().manual_seed(3)
    shapes, lrs = [(500, 3), (500, 15, 3), (500, 1)], [1.6e-4, 2.5e-3 / 20, 5e-2]
    params = [torch.randn(s, generator=g).numpy() for s in shapes]

    def grads_for_step(step):
        gg = torch.Generator().manual_seed(100 + step)
        gs = [torch.randn(s, generator=gg) * (0.0 if (step == 3 and i == 0) else 1e-3) for i, s in enumerate(shapes)]
        gs[1][::2] = 0.0
        return [t.numpy() for t in gs]
    return params, lrs, grads_for_step, {5: [(0, 1.0e-4)]}

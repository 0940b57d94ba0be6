#!/usr/bin/env python3
"""bench.py — fwd+bwd views/sec of the rasterizer hot path (BASELINE.json metric) on N B200s.

  python bench.py --gpus 1 --steps 50 --warmup 10                      # our kernels
  python bench.py --impl reference --gpus 1 --steps 20 --warmup 3      # reference CUDA kernels
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W        # one rank per GPU

A "step" is one full forward + backward of the differentiable rasterizer for one view per GPU
(1M Gaussians, 800x800, S=5 feature channels, SH degree 3, seeded synthetic `shell-v1` scene,
8-camera ring, fixed random cotangents); with N GPUs the views of a step are sharded one per GPU
and a single NCCL all-reduce of the per-Gaussian parameter gradients follows backward (weak
scaling).  Prints ONE JSON line on rank 0.

Keys: `value` = whole-job views/s with inputs resident in HBM (C-ABI level operator calls);
`e2e` = the same step through the reference-facing public API (GaussianRasterizer module +
autograd) including, every step, the host->device copy of that step's inputs from pinned memory
(camera + ground-truth image) and the device->host read of the loss; `roofline` = dominant kernel
vs the measured HBM peak (MEASURED_PEAKS.json); `cpu_baseline` = the CPU oracle port timed on a
bounded sample (rank 0, N=1 only).  `--impl reference` times the UNMODIFIED reference CUDA kernels
(oracle/_ref, built from /root/reference by oracle/build_ref.sh) on the same GPU; when that build
is absent it falls back to the CPU oracle port.
"""
import argparse
import ctypes
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HEADLINE = dict(P=1_000_000, W=800, H=800, S=5, views=8, recipe="shell-v1", seed=0)
# DRAM bytes per launch of the compositors at the headline config, from ncu --set full (profiles/)
NCU_TRAFFIC = {"composite_bwd": 63854848 + 1705728, "composite_fwd": 48878592 + 4990208}
STAGES = ["project", "depth_sort", "bin_count", "bin_offsets", "bin_scatter", "composite_fwd",   # bin_scatter includes tile_order + block_mask
          "surface_normal", "composite_bwd", "project_bwd"]


class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


def alg_bytes(P, Pv, R, HW, T, S):
    """Algorithmic bytes per stage and view (BASELINE.md §2.4; R, Pv measured in this run)."""
    ch = min(2048, max(512, -(-(-(-P // 444)) // 256) * 256))          # bin_chunk_len (csrc/common.cuh)
    chunks = -(-P // ch)
    return {
        "project": 236 * P + 48 * Pv,
        # depth-ordered binning (DESIGN.md section 4): 3 x (read + write) of P (key, id) pairs + first-pass count
        # read; walks over (id, rect) of the depth-sorted Gaussians; the chunk x tile matrix M
        "depth_sort": 52 * P, "bin_count": 12 * P + 4 * T * chunks,
        "bin_offsets": 12 * T * chunks + 12 * T,
        "bin_scatter": 24 * P + 4 * T * chunks + 4 * R,
        "composite_fwd": R * (4 + 40 + 4 * S) + HW * 4 * (3 + 1 + 1 + S) + 8 * HW + 4 * P,
        "surface_normal": 44 * HW,
        "composite_bwd": R * (44 + 4 * S) + HW * 4 * (5 + S) + 8 * HW + Pv * 4 * (11 + S),
        "project_bwd": Pv * (236 + 24 + 3 + 4 + 40) + P * 4 * (3 + 6 + 48 + 3 + 4),
    }


def workload_config(cfg, num_rendered):
    """The workload description — identical in both arms (arm-specific details live under "arm")."""
    return {"workload": f"rasterizer fwd+bwd, {cfg['recipe']} seed {cfg['seed']}, P={cfg['P']}, {cfg['W']}x{cfg['H']}, S={cfg['S']}, SH deg 3, "
                        f"{cfg['views']}-camera ring, one view per GPU per step, fixed random cotangents",
            "P": cfg["P"], "W": cfg["W"], "H": cfg["H"], "S": cfg["S"], "num_rendered": num_rendered,
            "l2": "inputs larger than L2 (236 MB Gaussian parameters + ~190 MB binning per step vs 126 MB L2)"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_inputs(cfg, device):
    from relightable3dgaussian_b200 import synth
    sc = synth.make_scene(cfg["P"], cfg["recipe"], cfg["seed"], cfg["S"])
    cams = [synth.make_camera(k, cfg["W"], cfg["H"]) for k in range(cfg["views"])]
    g = torch.Generator().manual_seed(1234)
    H, W, S = cfg["H"], cfg["W"], cfg["S"]
    cot = dict(color=torch.randn(3, H, W, generator=g), opacity=torch.randn(1, H, W, generator=g),
               depth=torch.randn(1, H, W, generator=g), feature=torch.randn(S, H, W, generator=g))
    gts = [torch.rand(3, H, W, generator=g) for _ in range(cfg["views"])]
    return sc, cams, cot, gts


def bench_ours(args, cfg, rank, local, world):
    from relightable3dgaussian_b200 import _C_raster as C, _lib, dist as rdist
    from relightable3dgaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer, set_deferred_count, set_grad_exchange
    import torch.distributed as tdist
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    sc, cams, cot, gts = make_inputs(cfg, dev)
    P, S, W, H = cfg["P"], cfg["S"], cfg["W"], cfg["H"]
    M = 16
    d = lambda t: t.to(dev)
    means3D, scales, rots, opac, shs, feats = map(d, (sc.means3D, sc.scales, sc.rotations, sc.opacities, sc.shs, sc.features))
    bg = torch.tensor([0.0, 0.0, 0.0], device=dev)
    camd = [dict(view=d(c.viewmatrix), proj=d(c.projmatrix), pos=d(c.campos), c=c) for c in cams]
    dcot = {k: d(v) for k, v in cot.items()}
    E = torch.Tensor([])
    # exchange step (N > 1): dense = one all-reduce of all per-Gaussian gradients (256 MB); factored = all-reduce
    # of the dense rest (64 MB) + all-gather of the rank-1 SH-gradient factors (12 MB per rank) + local rebuild
    factored = world > 1 and args.exchange in ("factored", "p2p", "auto")
    bucket, exchange_kind = None, "dense"
    if world > 1 and args.exchange in ("p2p", "auto"):
        try:                                             # one-kernel NVLink exchange; needs symmetric memory on this box
            bucket, exchange_kind = rdist.P2PGradExchange(P, S, M, dev), "p2p"
        except Exception as e:
            if args.exchange == "p2p":
                raise
            print(f"[bench] P2P exchange unavailable ({type(e).__name__}: {e}); using the NCCL factored exchange", file=sys.stderr)
    if bucket is None:
        bucket = rdist.FactoredGradExchange(P, S, M, dev) if factored else rdist.GradBucket(P, S, M, dev)
        exchange_kind = "factored" if factored else "dense"
    campos_tab = {}

    def campos_all(i):      # camera centres of the views the ranks render in step i, rank order
        key = (i * world) % cfg["views"]
        if key not in campos_tab:
            campos_tab[key] = torch.stack([camd[rdist.view_for_rank(i, r, world, cfg["views"])]["pos"] for r in range(world)]).contiguous()
        return campos_tab[key]
    stats = {}

    def step_resident(i):
        cam = camd[rdist.view_for_rank(i, rank, world, cfg["views"])]
        c = cam["c"]
        out = C.rasterize_gaussians(bg, means3D, feats, E, opac, scales, rots, 1.0, E, cam["view"], cam["proj"],
                                    c.tanfovx, c.tanfovy, c.cx, c.cy, H, W, shs, 3, cam["pos"], False, True, False)
        stats["R"] = out[0]; stats["radii"] = out[9]; stats["out"] = out
        C.rasterize_gaussians_backward(bg, means3D, feats, out[9], E, scales, rots, 1.0, E, cam["view"], cam["proj"],
                                       c.tanfovx, c.tanfovy, dcot["color"], dcot["opacity"], dcot["depth"],
                                       dcot["feature"], shs, 3, cam["pos"], out[10], out[0], out[11], out[12],
                                       True, False, _out=bucket.views)
        if factored:
            bucket.exchange(means3D, campos_all(i), 3)
        else:
            bucket.allreduce_mean()

    def timed(fn, steps, warmup, profile=False):
        for i in range(warmup):
            fn(i)
        # as timeit does: no collector inside the timed region — a pause in ONE of the N host processes stalls every rank
        # at the exchange.  Collected BEFORE the barrier, so that the ranks still enter the region together.
        gc.collect()
        gc.disable()
        if profile:
            lib.r3dg_prof_begin(steps)
        torch.cuda.synchronize(dev)
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(dev)
        l0 = lib.r3dg_launch_count()
        # the contract's timed region is the whole K steps (e0..e1); events between 5 equal blocks (no
        # synchronisation) additionally give a median-of-blocks figure that is robust to a one-off hiccup
        nblk = 5 if steps >= 10 else 1
        cuts = [steps * b // nblk for b in range(nblk + 1)]
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(nblk + 1)]
        evs[0].record()
        for b in range(nblk):
            for i in range(cuts[b], cuts[b + 1]):
                fn(warmup + i)
            evs[b + 1].record()
        gc.enable()
        torch.cuda.synchronize(dev)
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(dev)
        ms = evs[0].elapsed_time(evs[-1])
        blocks = [evs[b].elapsed_time(evs[b + 1]) / max(cuts[b + 1] - cuts[b], 1) for b in range(nblk)]
        stage = None
        if profile:
            arr = (ctypes.c_float * 9)(); nf = ctypes.c_int(); nb = ctypes.c_int()
            lib.r3dg_prof_end(arr, ctypes.byref(nf), ctypes.byref(nb))
            stage = {n: arr[i] / max(nf.value if i < 7 else nb.value, 1) for i, n in enumerate(STAGES)}
        launches = lib.r3dg_launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
            ms = float(t.item())
        stats["blocks"] = blocks
        return ms, stage, launches

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, stage, launches = timed(step_resident, args.steps, args.warmup, profile=True)
    blocks = stats["blocks"]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats["out"], bucket.views)
    value = world * args.steps / (ms / 1e3)

    # ---- e2e: public API (module + autograd), per-step host inputs from pinned memory -------
    params = [t.clone().requires_grad_(True) for t in (means3D, opac, shs, scales, rots, feats)]
    pinned_gt = [g.pin_memory() for g in gts]
    pinned_cam = [torch.cat([c.viewmatrix.reshape(-1), c.projmatrix.reshape(-1), c.campos]).pin_memory() for c in cams]
    # double-buffered device inputs: the H2D copy of step i+1 is issued on a copy stream while step i
    # computes (every step still copies its own inputs from pinned host memory inside the timed region)
    gt_dev = [torch.empty(3, H, W, device=dev) for _ in range(2)]
    cam_dev = [torch.empty(35, device=dev) for _ in range(2)]
    loss_host = torch.zeros(64).pin_memory()
    h2d = gt_dev[0].numel() * 4 + cam_dev[0].numel() * 4
    d2h = 4
    copy_stream = torch.cuda.Stream(device=dev)
    ready_ev = [torch.cuda.Event() for _ in range(2)]
    free_ev = [torch.cuda.Event() for _ in range(2)]
    pre = {"issued": None}

    def issue_copy(i):
        slot = i % 2
        v = rdist.view_for_rank(i, rank, world, cfg["views"])
        copy_stream.wait_event(free_ev[slot])              # the step that last read this slot has finished
        with torch.cuda.stream(copy_stream):
            gt_dev[slot].copy_(pinned_gt[v], non_blocking=True)
            cam_dev[slot].copy_(pinned_cam[v], non_blocking=True)
            ready_ev[slot].record(copy_stream)
        pre["issued"] = i

    def step_e2e(i):
        if pre["issued"] != i:                             # very first call only
            issue_copy(i)
        slot = i % 2
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready_ev[slot])
        c = cams[rdist.view_for_rank(i, rank, world, cfg["views"])]
        cd, gd = cam_dev[slot], gt_dev[slot]
        rs = GaussianRasterizationSettings(H, W, c.tanfovx, c.tanfovy, c.cx, c.cy, bg, 1.0,
                                           cd[:16].view(4, 4), cd[16:32].view(4, 4), 3, cd[32:35],
                                           False, True, True, False)
        p_means, p_opac, p_shs, p_scales, p_rots, p_feats = params
        means2D = torch.zeros_like(p_means, requires_grad=True)
        out = GaussianRasterizer(rs)(means3D=p_means, means2D=means2D, opacities=p_opac, shs=p_shs,
                                     scales=p_scales, rotations=p_rots, features=p_feats)
        issue_copy(i + 1)                                  # next step's inputs travel while this step computes
        color, opacity, depth, feature = out[2], out[3], out[4], out[5]
        loss = (color - gd).abs().mean() + 0.01 * opacity.mean() + 0.01 * depth.mean() + 0.01 * feature.square().mean()
        if leaf_bucket is not None:
            leaf_bucket.zero()                              # the dense rest accumulates straight into the flat all-reduce buffer
            p_shs.grad = None
            set_grad_exchange(bucket, campos_all(i))       # backward gathers the SH factors and rebuilds mean_v(dL_dsh)
        else:
            for p_ in params:
                p_.grad = None
        loss.backward()
        free_ev[slot].record(cur)
        if leaf_bucket is not None:
            leaf_bucket.allreduce_mean()                    # everything but SH is averaged at the leaves (one 64 MB all-reduce)
        elif world > 1:
            for p_ in params:                               # averaged in place, largest (SH, 192 MB) first in flight
                tdist.all_reduce(p_.grad, op=tdist.ReduceOp.AVG)
        loss_host[i % 64:i % 64 + 1].copy_(loss.detach().reshape(1), non_blocking=True)

    leaf_bucket = rdist.LeafGradBucket([params[k] for k in (0, 1, 3, 4, 5)], dev, symmetric=exchange_kind == "p2p") if factored else None
    e_steps = args.steps
    # (1) the path an UNCHANGED caller of the reference surface gets: synchronous instance count (one host wait per forward,
    #     like the reference's own cudaMemcpy at rasterizer_impl.cu:291).  Its warm-up also teaches the deferred path the counts.
    set_deferred_count(False)
    ms_sync, _, _ = timed(step_e2e, e_steps, max(min(args.warmup, 3), 3))
    # (2) opt-in: set_deferred_count(True) — no host round trip between forward and backward
    set_deferred_count(True)
    ms_e, _, _ = timed(step_e2e, e_steps, 8)
    set_deferred_count(False)
    set_grad_exchange(None)
    e2e_value = world * e_steps / (ms_sync / 1e3)
    e2e_deferred = world * e_steps / (ms_e / 1e3)

    res = None
    if rank == 0:
        Pv = int((stats["radii"] > 0).sum().item())
        R = int(stats["R"])
        T = ((W + 15) // 16) * ((H + 15) // 16)
        ab = alg_bytes(P, Pv, R, H * W, T, S)
        dom = max(stage, key=lambda k: stage[k])
        peak, peak_src = measured_peak()
        achieved = ab[dom] / (stage[dom] * 1e-3) / 1e9
        step_alg = sum(ab.values())
        res = {
            "metric": "fwd+bwd views/sec at 1M Gaussians 800x800, 1/2/4/8 B200; HBM GB/s vs peak" if cfg == HEADLINE else "fwd+bwd views/sec (non-headline config)",
            "value": value, "unit": "views/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "ms_per_step_block_median": statistics.median(blocks),
            "ms_per_step_blocks": blocks, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, R),
            "arm": {"impl": "relightable3dgaussian_b200 (libr3dg_b200.so through the C ABI)", "P_visible": Pv,
                    "exchange": exchange_kind if world > 1 else None,
                    "parallelism": ("single GPU" if world == 1 else
                                    f"view-parallel x{world}, per step ONE kernel over NVLink peer memory: SH gradient rebuilt from the peers' {bucket.factor.numel() * 4 / 1e6:.0f} MB "
                                    f"factor buffers (P2P loads) + in-switch (multimem{'' if bucket.multicast else ' unavailable: peer load/store'}) all-reduce of {bucket.n_dense * 4 / 1e6:.0f} MB dense grads, "
                                    "two symmetric-memory barriers, no NCCL collective" if exchange_kind == "p2p" else
                                    f"view-parallel x{world}, per step 1 NCCL all-reduce of {bucket.dense.bytes() / 1e6:.0f} MB dense grads + 1 all-gather of "
                                    f"{bucket.factor.numel() * 4 / 1e6:.0f} MB SH-gradient factors per rank + local rebuild" if exchange_kind == "factored" else
                                    f"view-parallel x{world}, 1 NCCL all-reduce of {bucket.bytes() / 1e6:.0f} MB grads/step")},
            "e2e": {"value": e2e_value, "unit": "views/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e_steps, "ms_per_step": ms_sync / e_steps,
                    "what": "GaussianRasterizer module exactly as an unchanged caller of the reference surface uses it (synchronous instance count) + autograd + L1 loss; "
                            "per step H2D of ground-truth image + camera from pinned memory (double-buffered, copy stream overlapping the previous step), D2H of the loss",
                    "deferred_count_opt_in": {"value": e2e_deferred, "ms_per_step": ms_e / e_steps,
                                              "what": "same, with rasterizer.set_deferred_count(True): the count is resolved in backward, no host round trip mid-step"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "stage_ms": stage,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": NCU_TRAFFIC.get(dom) if cfg == HEADLINE else None,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture per launch (profiles/r02_ncu_composite_*_final.md)",
                         "peak_source": peak_src,
                         "alg_bytes_per_launch": ab[dom],
                         "step_alg_bytes": step_alg, "step_frac_of_peak": step_alg / (ms / args.steps * 1e-3) / 1e9 / peak},
        }
    return res


DUMP_ROWS = 32768         # per-Gaussian outputs: a fixed, seeded sample of this many Gaussians (rows)


def dump_outputs(outdir, out, grads):
    """What the timed step returned in its last step, as <outdir>/<name>.npy: the rendered images and the per-pixel
    contributor counts whole, the per-Gaussian outputs (radii, weights, parameter gradients) on a seeded sample of
    DUMP_ROWS Gaussians (their indices in sample_rows.npy).  Float32 as computed; integers as float64 (exact)."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    P = out[9].shape[0]
    rows = np.sort(np.random.default_rng(0).choice(P, size=min(P, DUMP_ROWS), replace=False))
    rows_dev = torch.from_numpy(rows).to(out[9].device)
    arrays = {"num_rendered": np.array([int(out[0])], np.float64), "sample_rows": rows.astype(np.float64),
              "n_contrib": out[1].cpu().numpy().astype(np.float64), "radii": out[9][rows_dev].cpu().numpy().astype(np.float64)}
    for i, name in enumerate(("color", "opacity", "depth", "feature", "normal", "surface_xyz", "weights"), start=2):
        t = out[i] if name != "weights" else out[i][rows_dev]
        arrays[name] = t.float().cpu().numpy()
    for name, t in grads.items():
        arrays["grad_" + name] = t[rows_dev].float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise SystemExit(f"--dump-outputs: {total / 2**20:.1f} MB exceeds 64 MB at this configuration")
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)


def cpu_baseline_sample(cfg, seconds_budget=25.0):
    """The CPU oracle (port of the reference algorithm) on a bounded sample of the same workload: ONE full view —
    all P Gaussians at the full resolution, forward + backward — no extrapolation.  (Measured here: ~5-15 s for
    the headline config on the box's host cores.)"""
    import numpy as np
    from oracle import oracle
    from relightable3dgaussian_b200 import synth
    sc = synth.make_scene(cfg["P"], cfg["recipe"], cfg["seed"], cfg["S"])
    cam = synth.make_camera(0, cfg["W"], cfg["H"])
    n = lambda t: t.numpy()
    W, H, S = cfg["W"], cfg["H"], cfg["S"]
    rng = np.random.default_rng(0)
    cots = [rng.standard_normal((c, H, W)).astype(np.float32) for c in (3, 1, 1, S)]
    bg = np.zeros(3, np.float32)
    t0 = time.time()
    f = oracle.rasterize_forward(n(sc.means3D), n(sc.opacities), cam.viewmatrix.numpy(), cam.projmatrix.numpy(),
                                 cam.campos.numpy(), bg, W, H, cam.tanfovx, cam.tanfovy, cam.cx, cam.cy,
                                 shs=n(sc.shs), scales=n(sc.scales), rotations=n(sc.rotations), features=n(sc.features))
    oracle.rasterize_backward(f, n(sc.means3D), cam.viewmatrix.numpy(), cam.projmatrix.numpy(), cam.campos.numpy(), bg,
                              W, H, cam.tanfovx, cam.tanfovy, *cots, shs=n(sc.shs), scales=n(sc.scales),
                              rotations=n(sc.rotations), features=n(sc.features))
    dt = time.time() - t0
    return {"value": 1.0 / dt, "unit": "views/s", "cores": oracle.num_threads(), "kind": "port",
            "sample": f"1 complete view (fwd+bwd) of the full workload: all {cfg['P']} Gaussians at {W}x{H} (R={f['binned']['num_rendered']}) "
                      f"took {dt:.2f}s on {oracle.num_threads()} threads (C + OpenMP oracle); no extrapolation",
            "sample_seconds": dt}


def bench_reference(args, cfg, rank, local, world):
    """--impl reference: the unmodified reference CUDA kernels on this GPU (rank 0 only)."""
    if rank != 0:
        return None
    from oracle import ref_gpu
    base = {"impl": "reference", "metric": "fwd+bwd views/sec at 1M Gaussians 800x800, 1/2/4/8 B200; HBM GB/s vs peak" if cfg == HEADLINE else "fwd+bwd views/sec (non-headline config)",
            "unit": "views/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    P, S, W, H = cfg["P"], cfg["S"], cfg["W"], cfg["H"]
    if ref_gpu.available():
        dev = torch.device("cuda", local)
        torch.cuda.set_device(dev)
        sc, cams, cot, gts = make_inputs(cfg, dev)
        d = lambda t: t.to(dev)
        bg = torch.zeros(3, device=dev)
        dc = {k: d(v) for k, v in cot.items()}
        camd = [dict(view=d(c.viewmatrix), proj=d(c.projmatrix), pos=d(c.campos)) for c in cams]
        if ref_gpu.ext_available("raster") and not args.ref_shim:
            # STOCK code path: the reference's own Python wrapper -> its pybind module -> rasterize_points.cu -> its kernels,
            # forward + autograd backward with the same fixed cotangents
            raster, kind = ref_gpu.reference_rasterizer()
            leaves = [d(t).requires_grad_(True) for t in (sc.means3D, sc.opacities, sc.shs, sc.scales, sc.rotations, sc.features)]

            def step(i):
                c, cd = cams[i % len(cams)], camd[i % len(cams)]
                o = raster(c, cd, bg, *leaves)
                for t in leaves:
                    t.grad = None
                torch.autograd.backward([o["color"], o["opacity"], o["depth"], o["feature"]],
                                        [dc["color"], dc["opacity"], dc["depth"], dc["feature"]])
                return o
        else:
            kind = "reference CUDA kernels + rasterizer_impl.cu behind the raw-pointer shim (oracle/ref_shim_raster.cu)"
            kw = dict(means3D=d(sc.means3D), opacities=d(sc.opacities), shs=d(sc.shs), scales=d(sc.scales),
                      rotations=d(sc.rotations), features=d(sc.features))
            camk = [dict(viewmatrix=cd["view"], projmatrix=cd["proj"], campos=cd["pos"]) for cd in camd]
            ref = ref_gpu.RefRasterizer()

            def step(i):
                c, cd = cams[i % len(cams)], camk[i % len(cams)]
                o = ref.forward(bg=bg, W=W, H=H, tan_fovx=c.tanfovx, tan_fovy=c.tanfovy, cx=c.cx, cy=c.cy, **cd, **kw)
                ref.backward(o, bg=bg, tan_fovx=c.tanfovx, tan_fovy=c.tanfovy, dL_dcolor=dc["color"], dL_dopacity=dc["opacity"],
                             dL_ddepth=dc["depth"], dL_dfeature=dc["feature"], **cd,
                             **{k: v for k, v in kw.items() if k != "opacities"})
                return o
        for i in range(args.warmup):
            step(i)
        torch.cuda.synchronize()
        sampler = ClockSampler(local); sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gc.collect()
        gc.disable()          # both arms are timed the same way
        e0.record()
        for i in range(args.steps):
            o = step(args.warmup + i)
        e1.record()
        gc.enable()
        torch.cuda.synchronize()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1)
        v = args.steps / (ms / 1e3)
        base.update({"value": v, "ms_per_step": ms / args.steps, "clocks": clocks,
                     "config": workload_config(cfg, int(o["num_rendered"])),
                     "arm": {"impl": f"{kind}; sm_100 build of /root/reference, same scene / cameras / cotangents"},
                     "cpu_baseline": {"value": v, "unit": "views/s", "cores": os.cpu_count(), "kind": "reference",
                                      "sample": "not a CPU run: the reference has no CPU rasterizer; this is its own CUDA build timed on the same B200 (north_star), full workload, 8-camera ring"},
                     "e2e": {"value": v, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return base
    # fallback: CPU oracle port on a bounded sample
    cb = cpu_baseline_sample(cfg)
    base.update({"value": cb["value"], "ms_per_step": 1e3 / cb["value"],
                 "config": {"workload": "CPU oracle port of the reference algorithm (oracle/_ref CUDA build absent)"},
                 "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    return base


def main():
    # Only the JSON line may reach stdout: libraries (e.g. NCCL's version banner) print there too,
    # so fd 1 is pointed at stderr for the whole run and the result is written to the saved fd.
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 30 for --workload stage2)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--P", type=int, default=None)
    ap.add_argument("--W", type=int, default=None)
    ap.add_argument("--H", type=int, default=None)
    ap.add_argument("--S", type=int, default=None)
    ap.add_argument("--N", type=int, default=None, help="stage2: incident samples per Gaussian (default 32, script/run_dtu.sh:42)")
    ap.add_argument("--workload", default="headline", choices=["headline", "stage2"],
                    help="headline = BASELINE.json metric (rasterizer fwd+bwd, 1M / 800x800); stage2 = the neilf training step at BASELINE "
                         "configs #4 (1 GPU: 1.5M / 1600x1200) / #5 (N GPUs: 2M / 1920x1080), printed with \"workload\": \"stage2\"")
    ap.add_argument("--ref-shim", action="store_true", help="reference arm: force the raw-pointer shim instead of the stock wrapper + pybind module")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "factored", "dense"],
                    help="N > 1: gradient exchange per step (DESIGN.md section 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (headline workload, ours)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "headline"):
        ap.error("--dump-outputs applies to the headline workload of --impl ours")
    if args.steps is None:
        args.steps = 30 if args.workload == "stage2" else 200     # a stage-2 step is ~10x a headline step
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    args.warmup = max(args.warmup, 3)
    cfg = dict(HEADLINE)
    for k in ("P", "W", "H", "S"):
        if getattr(args, k) is not None:
            cfg[k] = getattr(args, k)
    from relightable3dgaussian_b200 import dist as rdist
    rank, local, world = rdist.init_from_env()
    if args.workload == "stage2":
        import bench_stage2
        cfg2 = dict(bench_stage2.CONFIG5 if world > 1 else bench_stage2.CONFIG4)
        for k in ("P", "W", "H", "N"):
            if getattr(args, k) is not None:
                cfg2[k] = getattr(args, k)
        if args.impl == "reference":
            if rank == 0:
                emit(bench_stage2.run_reference(args, cfg2, rank, local, world))
            if world > 1:
                import torch.distributed as tdist
                tdist.barrier()
                tdist.destroy_process_group()
            return
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA GPU: the hot path has no CPU fallback")
        res = bench_stage2.run_ours(args, cfg2, rank, local, world)
        if rank == 0:
            emit(res)
        if world > 1:
            import torch.distributed as tdist
            tdist.barrier()
            tdist.destroy_process_group()
        return
    if args.impl == "reference":
        if rank == 0:
            emit(bench_reference(args, cfg, rank, local, world))
        if world > 1:                      # the other ranks do no work; leave the group together
            import torch.distributed as tdist
            tdist.barrier()
            tdist.destroy_process_group()
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA GPU: the rasterizer hot path has no CPU fallback")
    res = bench_ours(args, cfg, rank, local, world)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                res["cpu_baseline"] = cpu_baseline_sample(cfg)
            except Exception as e:   # the oracle is only a reported baseline
                res["cpu_baseline"] = {"value": None, "unit": "views/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        emit(res)
    if world > 1:
        import torch.distributed as tdist
        tdist.barrier()
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()

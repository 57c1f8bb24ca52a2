#!/usr/bin/env python
"""bench.py -- fwd+bwd views/sec of the surfel-rasterizer hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json north_star point): synthetic ``scene(131072, seed 0)`` (SURVEY 8d),
512x512, white background, degree-1 SH, LaRa-like upstream gradients; every rank renders
`--views` (default 8) target views per step, forward AND backward.  View-sharded weak
scaling: N ranks -> N*views distinct views per step over the same Gaussian set, parameter
gradients summed per rank inside the per-Gaussian backward and across ranks with a single NCCL
all-reduce per step.  A "step" = those fwd+bwd views + the all-reduce.

Printed JSON (one line, rank 0):
  value   : views/s, whole job, inputs resident in HBM, through lara_b200.sharded.render_views
            (the batched srf_views_* launch set: every kernel carries a view dimension; per-step
            CUDA events on the launching stream, L2 flushed between steps outside the timed spans,
            max over ranks)
  e2e     : the same metric through the reference-facing drop-in API
            (diff_surfel_rasterization.GaussianRasterizer + autograd, ONE VIEW PER CALL exactly like
            the reference arm), with the Gaussian parameters and cameras copied from pinned host memory
            every step and the summed parameter gradients read back to the host every step;
            e2e.batched is the same host-in / host-out protocol through the batched public entry
            (lara_b200.multiview.render_scene_views, one autograd node per scene)
  roofline: dominant kernel (render_bwd) -- SURVEY 8d algorithmic bytes per launch / its live
            CUDA-event duration (srf_profile_*), against MEASURED_PEAKS.json hbm_gbs; roofline.issue states
            the bound that actually binds the blend kernels (warp-instruction issue slots)
  extra   : BASELINE configs C2 (32k / 512^2 / 1 view), C4 (256k / 1024^2, 4 views per GPU), the strong-scaling
            point (8 global views split over the ranks) and a >= 2 s sustained run
  grad_check (N > 1): rank 0 re-renders all N*V views alone and compares with the all-reduced buffer
  cpu_baseline: the CPU oracle port (oracle/surfel_oracle.c, OpenMP) on a bounded sample of the same
            workload (N=1, rank 0 only)
--impl reference times the reference's own CUDA build (oracle/_ref) through its own Python
API on one GPU (rank 0), same workload and extras; the reference has no CPU rasterizer.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "rasterizer fwd+bwd views/sec at {P} Gaussians x {S}x{S}"      # formatted with --P / --size (defaults: the north-star point)
UNIT = "views/s"
PARAM_KEYS = ("means3D", "shs", "opacities", "scales", "rotations")
# batched launch set per step: preprocess_fwd, tile_scan, scatter, sort_small, sort_big, render_fwd, render_bwd, preprocess_bwd
KERNELS_PER_STEP = 8


def workload_string(P, size, views):
    return f"scene({P},seed0) {size}x{size} sh1 white bg, {views} views/GPU/step fwd+bwd"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--views", type=int, default=8, help="target views per GPU per step")
    ap.add_argument("--P", type=int, default=131072)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra configurations (C2, C4, strong point, sustained)")
    ap.add_argument("--streams", type=int, default=1, help="ignored (the views of a step share one launch set)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (images, aux maps, radii, parameter gradients) "
                         "as DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path only")
    return args


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (rank 0)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], None, set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None}


def dist_info():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def timed_steps(step_fn, steps, warmup, flush, world, dev):
    """W untimed + K timed steps; per-step CUDA events, L2 flush between steps (untimed).
    Returns (ms summed over the K steps: max over ranks, (min, max) over ranks of that sum)."""
    import torch.distributed as dist
    for _ in range(warmup):
        flush.zero_()
        step_fn()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()               # evict the previous step's working set from the 126 MB L2
        starts[i].record()
        step_fn()
        ends[i].record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    spread = (ms, ms)
    if world > 1:
        t = torch.tensor([ms, -ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        spread = (-float(t[1].item()), float(t[0].item()))
        ms = float(t[0].item())
    return ms, spread


def dump_outputs(out_dir, arrays, budget=64 * 10**6):
    """Writes each tensor as float32 ``out_dir/<name>.npy``.  Smaller tensors are written whole; one larger than
    an equal share of the budget still left is replaced by a fixed, seeded sample of its flattened elements
    (in index order), so that two builds given the same arguments write comparable files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = budget - 256 * len(items)                     # room for the .npy headers
    for i, (name, t) in enumerate(items):
        a = t.detach().float().cpu().numpy()
        share = left // (len(items) - i) // 4
        if a.size > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= 4 * a.size


def cpu_baseline(P, size, budget_s=10.0, max_views=8):
    """Oracle port on the host cores: fwd+bwd views of the same workload until ~budget_s of CPU work."""
    from lara_b200 import scene as S
    from oracle import oracle as O
    sc = S.scene(P, 0, sh_degree=1)
    cams = S.cameras(8, size, size, 0)
    gc, ga = S.upstream_grads(size, size, 0, lara_like=True)
    O.load()
    t0 = time.perf_counter()
    n = 0
    while n < max_views and (n == 0 or time.perf_counter() - t0 < budget_s):
        run = O.run_scene(sc, cams[n % len(cams)], torch.ones(3))
        run.backward(gc, ga)
        run.close()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": O.threads(), "kind": "port",
            "sample": f"{n} view(s) fwd+bwd of the {P}-Gaussian {size}x{size} workload, CPU oracle (C + OpenMP), {dt:.1f} s"}


class Workload:
    """Resident inputs of one configuration: parameters, per-view settings, packed cameras, stacked upstream grads."""

    def __init__(self, P, size, view_ids, total_views, dev, settings_cls, seed=0):
        from lara_b200 import scene as S
        self.P, self.size, self.ids = P, size, list(view_ids)
        self.sc = S.scene(P, seed, sh_degree=1)
        self.cams = S.cameras(total_views, size, size, 0)
        gc, ga = S.upstream_grads(size, size, 0, lara_like=True)
        self.gc, self.ga = gc.to(dev), ga.to(dev)
        self.bg = torch.ones(3)
        self.params = {k: self.sc[k].to(dev) for k in PARAM_KEYS}
        self.M = int(self.params["shs"].shape[1])
        self.sets = [S.settings_for(self.cams[i], self.bg, 1, dev, settings_cls) for i in self.ids]
        self.dev = dev

    def stacked_grads(self):
        V = len(self.ids)
        return (self.gc.expand(V, -1, -1, -1).contiguous(), self.ga.expand(V, -1, -1, -1).contiguous())


def make_batched_step(wl, grads, all_reduce=True, coll_events=None):
    """One step through the batched launch set, inputs resident."""
    from lara_b200 import rasterizer as R, sharded
    packed = R.pack_cameras(wl.sets, wl.dev)
    G = wl.stacked_grads()

    def step():
        grads.zero_()
        # (color, allmap, radii) per view of the latest step, for --dump-outputs
        step.views, _ = sharded.render_views(wl.params, wl.sets, None, grads=grads, view_ids=wl.ids, cams=packed,
                                             upstream_stacked=G)
        if all_reduce:
            if coll_events is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); grads.all_reduce(); e1.record()
                coll_events.append((e0, e1))
            else:
                grads.all_reduce()
    return step


def make_dropin_step(wl, mod, host_io=None, world=1):
    """One step through a GaussianRasterizer-style API (`mod` = the drop-in package or the reference build),
    one view per call + autograd.  host_io = (pinned params, pinned cams [V,36], pinned out): parameters and
    cameras travel from pinned host memory and the summed gradients go back every step."""
    import torch.distributed as dist
    dev = wl.dev
    bg_dev = wl.bg.to(dev)
    if host_io is None:
        leaves = {k: wl.params[k].clone().requires_grad_(True) for k in PARAM_KEYS}
        m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)

        def step():
            for v in leaves.values():
                v.grad = None
            for rs in wl.sets:
                rast = mod.GaussianRasterizer(raster_settings=rs)
                c, rd, am = rast(means3D=leaves["means3D"], means2D=m2d, shs=leaves["shs"], opacities=leaves["opacities"],
                                 scales=leaves["scales"], rotations=leaves["rotations"])
                torch.autograd.backward((c, am), (wl.gc, wl.ga))
        return step

    pinned, cam_host, host_out = host_io

    def step_e2e():
        dp = {k: v.to(dev, non_blocking=True).requires_grad_(True) for k, v in pinned.items()}
        m2d = torch.zeros_like(dp["means3D"], requires_grad=True)
        cam_dev = cam_host.to(dev, non_blocking=True)
        for r_, i in enumerate(wl.ids):
            c = wl.cams[i]
            rs = mod.GaussianRasterizationSettings(
                image_height=c.image_height, image_width=c.image_width, tanfovx=c.tanfovx, tanfovy=c.tanfovy,
                bg=bg_dev, scale_modifier=1.0, viewmatrix=cam_dev[r_, 0:16].view(4, 4),
                projmatrix=cam_dev[r_, 16:32].view(4, 4), sh_degree=1, campos=cam_dev[r_, 32:35],
                prefiltered=False, debug=False)
            rast = mod.GaussianRasterizer(raster_settings=rs)
            color, radii, allmap = rast(means3D=dp["means3D"], means2D=m2d, shs=dp["shs"], opacities=dp["opacities"],
                                        scales=dp["scales"], rotations=dp["rotations"])
            torch.autograd.backward((color, allmap), (wl.gc, wl.ga))
        flat = torch.cat([dp[k].grad.reshape(-1) for k in PARAM_KEYS])
        if world > 1:
            dist.all_reduce(flat)
        host_out[:flat.numel()].copy_(flat, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()   # the caller reads the result
    return step_e2e


def make_batched_e2e_step(wl, host_io, world=1):
    """Host in / host out through the batched public entry (one autograd node, one launch set per scene)."""
    import torch.distributed as dist
    from lara_b200 import rasterizer as R
    from lara_b200.multiview import _RenderSceneViews, shared_view_settings
    dev = wl.dev
    pinned, cam_host, host_out = host_io
    V = len(wl.ids)
    G = wl.stacked_grads()
    bg_dev = wl.bg.to(dev)
    c0 = wl.cams[wl.ids[0]]

    class _RasterViews(torch.autograd.Function):
        """colour + aux maps of all views of one scene (the rasterizer half of render_scene_views)."""
        @staticmethod
        def forward(ctx, means3D, shs, opac, scales, rot, sets):
            H, W, tfx, tfy, deg, pre, dbg = shared_view_settings(sets)
            cams = R.pack_cameras(sets, dev)
            color, allmap, radii, state = R.forward_views_raw(means3D, shs, None, opac, scales, rot, None, cams, tfx, tfy, H, W, deg)
            ctx.save_for_backward(means3D, shs, scales, rot, cams, radii)
            ctx.state, ctx.geo = state, (H, W, tfx, tfy, deg)
            return color, allmap

        @staticmethod
        def backward(ctx, g_color, g_allmap):
            means3D, shs, scales, rot, cams, radii = ctx.saved_tensors
            H, W, tfx, tfy, deg = ctx.geo
            g = R.backward_views_raw(ctx.state, radii, means3D, shs, None, scales, rot, None, cams, tfx, tfy, H, W, deg,
                                     g_color.contiguous(), g_allmap.contiguous())
            return g["means3D"], g["sh"], g["opacities"], g["scales"], g["rotations"], None

    def step():
        dp = {k: v.to(dev, non_blocking=True).requires_grad_(True) for k, v in pinned.items()}
        cam_dev = cam_host.to(dev, non_blocking=True)
        sets = [R.GaussianRasterizationSettings(
            image_height=c0.image_height, image_width=c0.image_width, tanfovx=c0.tanfovx, tanfovy=c0.tanfovy,
            bg=bg_dev, scale_modifier=1.0, viewmatrix=cam_dev[r_, 0:16].view(4, 4), projmatrix=cam_dev[r_, 16:32].view(4, 4),
            sh_degree=1, campos=cam_dev[r_, 32:35], prefiltered=False, debug=False) for r_ in range(V)]
        # rasterizer outputs are what the upstream gradients are defined on: use the raw batched autograd node
        color_allmap = _RasterViews.apply(dp["means3D"], dp["shs"], dp["opacities"], dp["scales"], dp["rotations"], sets)
        torch.autograd.backward(color_allmap, G)
        flat = torch.cat([dp[k].grad.reshape(-1) for k in PARAM_KEYS])
        if world > 1:
            dist.all_reduce(flat)
        host_out[:flat.numel()].copy_(flat, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    return step


def host_buffers(wl, grads_numel):
    pinned = {k: wl.sc[k].pin_memory() for k in PARAM_KEYS}
    # all cameras of the step travel in one pinned buffer: [V, 16 view | 16 proj | 3 campos | pad]
    cam_host = torch.zeros((len(wl.ids), 36), dtype=torch.float32)
    for r_, i in enumerate(wl.ids):
        cam_host[r_, 0:16] = wl.cams[i].viewmatrix.reshape(-1)
        cam_host[r_, 16:32] = wl.cams[i].projmatrix.reshape(-1)
        cam_host[r_, 32:35] = wl.cams[i].campos
    cam_host = cam_host.pin_memory()
    host_out = torch.empty(grads_numel, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * 4 for t in pinned.values()) + cam_host.numel() * 4
    return (pinned, cam_host, host_out), h2d, host_out.numel() * 4


C3_SCENES = 8

EXTRA_CONFIGS = [      # name, P, size, views per GPU   (BASELINE.json configs[1] and configs[3])
    ("C2_32k_512_1view", 32768, 512, 1),
    ("C4_256k_1024_4views_per_gpu", 262144, 1024, 4),
]


def run_reference(args, rank, local, world):
    """Reference arm: the unmodified reference CUDA build through its own Python API, rank 0 only."""
    if rank != 0:
        return
    from oracle import ref as REF
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    base = {"impl": "reference", "metric": METRIC.format(P=args.P, S=args.size), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic"}
    if not REF.available():
        # the oracle always exists: fall back to the CPU port
        cb = cpu_baseline(args.P, args.size)
        base.update({"value": cb["value"], "ms_per_step": 1e3 / cb["value"], "cpu_baseline": cb,
                     "config": {"workload": workload_string(args.P, args.size, args.views),
                                "note": "oracle/_ref not built: CPU oracle port, bounded sample on the host cores"},
                     "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(base), flush=True)
        return
    ref = REF.load()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def measure(P, size, views, steps, warmup):
        wl = Workload(P, size, range(views), views, dev, ref.GaussianRasterizationSettings)
        step = make_dropin_step(wl, ref)
        ms, _ = timed_steps(step, steps, warmup, flush, 1, dev)
        return views * steps / (ms / 1e3), ms / steps

    sampler = ClockSampler(local)
    sampler.start()
    value, ms_step = measure(args.P, args.size, args.views, args.steps, max(args.warmup, 3))
    clocks = sampler.stop()
    extra = {}
    if not args.no_extra:
        for name, P, size, views in EXTRA_CONFIGS:
            v, m = measure(P, size, views, max(3, args.steps // 4), 3)
            extra[name] = {"value": v, "unit": UNIT, "ms_per_step": m, "views_per_step": views}
        v, m = measure(524288, 512, 8, 2, 1)              # one scene's 8 views; a step of C3 is 8 such scenes
        extra["C3_raster_share_524k_8views_per_scene"] = {"value": v, "unit": UNIT, "ms_per_step": m * C3_SCENES, "scenes_per_gpu": C3_SCENES,
                                                          "views_per_scene": 8, "note": "timed on one scene (8 views), step time scaled to 8 scenes"}
        v, m = measure(args.P, args.size, 8, max(3, args.steps // 2), 3)
        extra["strong_8_global_views"] = {"value": v, "unit": UNIT, "ms_per_step": m, "views_per_step": 8,
                                          "note": "the reference is single-GPU: all 8 views on one B200"}
    base.update({
        "value": value, "ms_per_step": ms_step,
        "config": {"workload": workload_string(args.P, args.size, args.views),
                   "api_level": "reference's GaussianRasterizer + autograd, one view per call, inputs resident, 1 B200",
                   "views_per_gpu": args.views, "l2": "flushed between steps (256 MiB write, untimed)"},
        "clocks": clocks,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                         "sample": "reference's own CUDA rasterizer (oracle/_ref) on 1 B200 -- the reference ships no CPU rasterizer"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "extra": extra,
    })
    print(json.dumps(base), flush=True)


def main():
    args = parse_args()
    rank, local, world = dist_info()
    if args.impl == "reference":
        run_reference(args, rank, local, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the rasterizer has no CPU path)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", device_id=dev)

    from lara_b200 import rasterizer as R
    from lara_b200 import sharded, _lib
    from lara_b200.debug import unpack_state
    import diff_surfel_rasterization as DSR   # the drop-in name LaRa imports

    _lib.load()
    V = args.views
    total_views = V * world
    my_ids = sharded.shard_views(total_views, rank, world)
    wl = Workload(args.P, args.size, my_ids, total_views, dev, R.GaussianRasterizationSettings)
    P, M = args.P, wl.M
    grads = sharded.GradBuffer(P, M, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    coll = []
    step = make_batched_step(wl, grads, all_reduce=True, coll_events=coll if world > 1 else None)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        flush.zero_(); step()
    torch.cuda.synchronize(dev)
    coll.clear()
    if sampler:
        sampler.start()
    ms, spread = timed_steps(step, args.steps, 0, flush, world, dev)
    value = total_views * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        outs = {"color": torch.stack([c for c, _, _ in step.views]), "allmap": torch.stack([a for _, a, _ in step.views]),
                "radii": torch.stack([r for _, _, r in step.views])}
        outs.update({"grad_" + k: v for k, v in grads.views.items()})
        dump_outputs(args.dump_outputs, outs)
    collective_us = None
    rank_compute_ms = None
    if coll:
        collective_us = 1e3 * sum(a.elapsed_time(b) for a, b in coll[-args.steps:]) / args.steps
        # per-rank time spent inside the all-reduce (transfer + waiting for the slowest rank), gathered from every rank:
        # the rank with the SMALLEST value is the one the others wait for
        mine = torch.tensor([collective_us], dtype=torch.float64, device=dev)
        allc = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allc, mine)
        rank_compute_ms = [round(ms / args.steps - float(c.item()) / 1e3, 4) for c in allc]   # step time minus own collective time
        collective_us = {"rank0": collective_us, "per_rank": [round(float(c.item()), 1) for c in allc]}

    # ---- hardware correctness of the sharded step: the all-reduced buffer equals the single-rank sum
    grad_check = None
    if world > 1:
        reduced = grads.flat.clone()
        if rank == 0:
            wl_all = Workload(args.P, args.size, range(total_views), total_views, dev, R.GaussianRasterizationSettings)
            g_all = sharded.GradBuffer(P, M, dev)
            make_batched_step(wl_all, g_all, all_reduce=False)()
            torch.cuda.synchronize(dev)
            scale = float(g_all.flat.abs().max().item())
            err = float((reduced - g_all.flat).abs().max().item()) / (scale if scale > 0 else 1.0)
            grad_check = {"status": "ok" if err < 1e-5 else "FAILED", "max_rel_err": err,
                          "what": f"all-reduced parameter gradients of {world} ranks x {V} views vs {total_views} views on rank 0"}
            del wl_all, g_all
        dist.barrier()

    # ---- end to end through the reference-facing API, host buffers in / gradients out
    host_io, h2d, d2h = host_buffers(wl, grads.flat.numel())
    e2e_steps = max(3, args.steps // 2)
    ms_e2e, _ = timed_steps(make_dropin_step(wl, DSR, host_io, world), e2e_steps, 3, flush, world, dev)
    e2e_value = total_views * e2e_steps / (ms_e2e / 1e3)
    ms_e2b, _ = timed_steps(make_batched_e2e_step(wl, host_io, world), e2e_steps, 3, flush, world, dev)
    e2e_batched = total_views * e2e_steps / (ms_e2b / 1e3)
    # the per-view drop-in API with resident inputs (no host copies): separates "one launch set per view" from the copies
    ms_dr, _ = timed_steps(make_dropin_step(wl, DSR), e2e_steps, 3, flush, world, dev)
    dropin_resident = total_views * e2e_steps / (ms_dr / 1e3)
    clocks = sampler.stop() if sampler else None

    # ---- extra configurations: C2, C4, strong-scaling point, sustained run
    extra = {}
    if not args.no_extra:
        for name, Pe, Se, Ve in EXTRA_CONFIGS:
            ids = sharded.shard_views(Ve * world, rank, world)
            wle = Workload(Pe, Se, ids, Ve * world, dev, R.GaussianRasterizationSettings)
            ge = sharded.GradBuffer(Pe, wle.M, dev)
            ks = max(3, args.steps // 4)
            m, _ = timed_steps(make_batched_step(wle, ge), ks, 3, flush, world, dev)
            entry = {"value": Ve * world * ks / (m / 1e3), "unit": UNIT, "ms_per_step": m / ks,
                     "views_per_step_global": Ve * world, "api_level": "batched srf_views_* launch set, inputs resident"}
            if Ve == 1:
                # the drop-in per-view API on the same configuration (latency of ONE GaussianRasterizer fwd+bwd)
                m2, _ = timed_steps(make_dropin_step(wle, DSR), 4 * ks, 5, flush, world, dev)
                entry["dropin_api_ms_per_view"] = m2 / (4 * ks)
            extra[name] = entry
            del wle, ge
        # C3 / C5 (BASELINE configs[2], [4]): the rasterizer share of a LaRa train step -- 8 target views per scene at LaRa's
        # own Gaussian count, 8 scenes on one GPU (C3) or 32 scenes over 8 GPUs = 4 per GPU (C5); scenes are data-parallel
        # (the DDP all-reduce of the NETWORK gradients is outside this path), so no collective inside the step
        n_sc = C3_SCENES if world == 1 else max(1, 32 // world)
        wls = [Workload(524288, 512, range(8), 8, dev, R.GaussianRasterizationSettings, seed=sd) for sd in range(min(n_sc, 2))]
        gsc = sharded.GradBuffer(524288, wls[0].M, dev)
        steps_sc = [make_batched_step(w_, gsc, all_reduce=False) for w_ in wls]

        def step_scenes():
            for k in range(n_sc):
                steps_sc[k % len(steps_sc)]()
        ks = max(2, args.steps // 5)
        m, _ = timed_steps(step_scenes, ks, 2, flush, world, dev)
        extra["C3_raster_share_524k_8views_per_scene"] = {
            "value": n_sc * 8 * world * ks / (m / 1e3), "unit": UNIT, "ms_per_step": m / ks, "scenes_per_gpu": n_sc,
            "views_per_scene": 8, "note": "rasterizer fwd+bwd share of the train step (network, loss and DDP all-reduce are outside the path)"}
        del wls, gsc, steps_sc
        if 8 % world == 0:
            ids = sharded.shard_views(8, rank, world)
            wls = Workload(args.P, args.size, ids, 8, dev, R.GaussianRasterizationSettings)
            gs = sharded.GradBuffer(P, M, dev)
            ks = max(3, args.steps // 2)
            m, _ = timed_steps(make_batched_step(wls, gs), ks, 3, flush, world, dev)
            extra["strong_8_global_views"] = {"value": 8 * ks / (m / 1e3), "unit": UNIT, "ms_per_step": m / ks,
                                              "views_per_gpu": 8 // world, "scaling": "strong"}
            del wls, gs
        # sustained: the main step back to back for >= 2 s, timed as one region (no L2 flush: the per-step working set
        # of 8 views' state is several times the 126 MB L2)
        n_sus = max(10, int(2.5 / (ms / 1e3 / args.steps)))
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_sus):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
        sus_ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([sus_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sus_ms = float(t.item())
        extra["sustained"] = {"value": total_views * n_sus / (sus_ms / 1e3), "unit": UNIT, "seconds": sus_ms / 1e3, "steps": n_sus}

    # ---- roofline of the dominant kernel (render_bwd), live CUDA-event timing of every launch
    roof = None
    kern = None
    prof_steps = min(args.steps, 5)
    if rank == 0:
        _lib.profile_begin()
    step_noreduce = make_batched_step(wl, grads, all_reduce=False)
    for _ in range(prof_steps):
        flush.zero_(); step_noreduce()
    torch.cuda.synchronize(dev)
    if rank == 0:
        kern = _lib.profile_end()
        # measured sizes of the rank's views for the algorithmic byte count (SURVEY 8d)
        color, allmap, radii, st = R.forward_views_raw(wl.params["means3D"], wl.params["shs"], None, wl.params["opacities"],
                                                       wl.params["scales"], wl.params["rotations"], None,
                                                       R.pack_cameras(wl.sets, dev), wl.sets[0].tanfovx, wl.sets[0].tanfovy,
                                                       args.size, args.size, 1)
        torch.cuda.synchronize(dev)
        gx = (args.size + 15) // 16
        r_eff_views, R_views = [], st.resolve()
        for v in range(len(my_ids)):
            u = unpack_state(st, P, args.size, args.size, view=v)
            ncon = u["n_contrib"][0][:gx * 16, :gx * 16] if args.size % 16 == 0 else None
            if ncon is None:
                continue
            ncon = ncon.reshape(gx, 16, gx, 16).permute(0, 2, 1, 3).reshape(gx * gx, 256)
            r_eff_views.append(int(ncon.max(dim=1).values.sum().item()))
        npix = args.size * args.size
        r_eff = sum(r_eff_views)
        nv = max(len(r_eff_views), 1)
        alg_bytes = 148 * r_eff + 64 * npix * nv          # K7: (76+72)*R_eff + 64*Npix per view  (SURVEY 8d), all views of the launch
        tot_ms, n_launch = kern["render_bwd"]
        dur_s = tot_ms / 1e3 / max(n_launch, 1)
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peak = float(json.load(f)["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
        traffic = warp_inst = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                if args.P == 131072 and args.size == 512:      # the capture is of the default workload only
                    j = json.load(f)
                    # the capture is of one kernel variant: a different one running now has no ncu figures
                    if int(j.get("bwd_variant", -1)) == _lib.select_bwd_variant(0):
                        traffic = j.get("render_bwd_dram_bytes_per_view")
                        if traffic is not None:
                            traffic = traffic * nv
                        warp_inst = j.get("render_bwd_warp_instructions_per_view")
        except Exception:
            pass
        achieved = alg_bytes / dur_s / 1e9
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        issue = None
        if warp_inst is not None:
            slots = 148 * 4 * sm_mhz * 1e6 * dur_s          # SMs x schedulers x clock x time
            issue = {"bound": "issue", "warp_instructions_per_launch": warp_inst * nv, "issue_slots": slots,
                     "frac": warp_inst * nv / slots, "source": "ncu smsp__inst_executed.sum of profiles/ (per view) x views per launch"}
        roof = {"kernel": "render_bwd_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "views_per_launch": nv, "R": R_views, "R_eff": r_eff_views,
                "avg_launch_us": dur_s * 1e6, "issue": issue,
                "note": "the blend kernels are fp32-issue bound, not HBM bound (DESIGN.md); per-kernel us per view in 'kernels_us'"}

    if rank == 0:
        nv = len(my_ids)
        out = {
            "metric": METRIC.format(P=args.P, S=args.size), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.P, args.size, V),
                       "api_level": "value: batched srf_views_* launch set (lara_b200.sharded.render_views), inputs resident; "
                                    "e2e: drop-in GaussianRasterizer + autograd, one view per call, pinned host in / grads out",
                       "views_per_gpu": V, "global_views_per_step": total_views,
                       "parallelism": f"view-shard x{world} + 1 NCCL all-reduce of param grads",
                       "l2": "flushed between steps (256 MiB write, untimed)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "diff_surfel_rasterization.GaussianRasterizer + autograd (one view per call), pinned host in / grads out",
                    "dropin_api_inputs_resident": {"value": dropin_resident, "unit": UNIT,
                                                   "api": "the same per-view autograd API without the host copies (what the reference arm measures)"},
                    "batched": {"value": e2e_batched, "unit": UNIT,
                                "api": "same host-in/host-out protocol, one autograd node + one launch set per scene (srf_views_*)"}},
            "gpu_launches": KERNELS_PER_STEP * args.steps * world,
            "clocks": clocks,
            "roofline": roof,
            "kernels_us": {k: (v[0] * 1e3 / v[1] / nv if v[1] else 0.0) for k, v in kern.items()} if kern else None,
            "rank_step_ms": {"min": spread[0] / args.steps, "max": spread[1] / args.steps},
            "collective_us": collective_us, "rank_compute_ms": rank_compute_ms,
            "grad_check": grad_check["status"] if grad_check else None,
            "grad_check_detail": grad_check,
            "extra": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args.P, args.size)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

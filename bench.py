#!/usr/bin/env python
"""bench.py -- views/sec of the rasterizer hot path on BASELINE.json's configurations.

  cfg3 (default; cfg4 = the same scene view-sharded over N GPUs): forward+backward, 1M Gaussians, 1920x1080.
      A "step" is one camera view: plugin render (attribute activations + rasterizer forward) -> loss on colour +
      depth + opacity -> backward -> depth->normal map.
  cfg5: forward only (no_grad), 5M Gaussians unbounded-scene-shaped, 1440x1080: depth + median depth + opacity +
      normal, the mesh / point-cloud extraction pass (extract_mesh.py:95-115, extract_pcd.py:314-345).
  --train 1: cfg3 as a data-parallel TRAINING step (SURVEY.md 8f row 3): every rank renders `--views-per-step`
      views, gradients are summed over ranks with bucketed all_reduces that overlap the remaining views of the
      step, then ONE fused AdamW launch (1/world scaling and zero_grad folded in).

One process per GPU (torchrun for N>1), views sharded k = rank (mod N), "weak" scaling: every rank does K steps.
Without --train the Gaussian-parameter gradients stay local and the only collective is one all_gather of the
per-view loss scalars at the end of the timed region.

  python bench.py --gpus N --steps K --warmup W            # this framework
  python bench.py --impl reference --gpus N ...            # the UNMODIFIED reference CUDA extension
                                                           # (oracle/_ref/_refC.so) driven by the same loop;
                                                           # loads nothing of this framework's native code
  python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed as
                                                           # DIR/<name>.npy, to compare two builds output for output

Prints ONE JSON line on rank 0 (see DESIGN.md, Measurement, for every key).
"""
import argparse
import ctypes
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

STAGES = ["preprocess_fwd", "tile_scan", "scatter", "tile_sort", "render_fwd", "render_bwd", "preprocess_bwd",
          "depth2normal"]
# init_header, preprocess_fwd, tile_scan, scatter, tile_sort x4 (size tiers), render_fwd, depth2normal (+ render_bwd,
# preprocess_bwd when there is a backward); the pixel-loss kernels are torch's and not counted
KERNELS_FWD, KERNELS_BWD = 10, 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="new", choices=["new", "reference"])
    ap.add_argument("--config", default="cfg3", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--sh-degree", type=int, default=None, help="active SH degree (cfg5 is also quoted at 0)")
    ap.add_argument("--gaussians", type=int, default=None, help="override P (debug only; invalidates the number)")
    ap.add_argument("--pipelined", type=int, default=1, help="sync-free forward (capacity from high-water mark)")
    ap.add_argument("--fused", type=int, default=1, help="fused activations inside the projection kernel")
    ap.add_argument("--streams", type=int, default=3,
                    help="independent views alternate over this many CUDA streams (the library is stream-aware; the "
                         "reference launches on the legacy default stream and cannot overlap views)")
    ap.add_argument("--graph", type=int, default=1,
                    help="replay each view's render(+loss+backward)+normal as one CUDA graph (gaustudio_b200.graphs)")
    ap.add_argument("--dropin", type=int, default=1,
                    help="also time the drop-in path exactly as gaustudio calls it (un-fused torch activations, exact "
                         "forward, one stream, eager) and report it as `dropin` (N=1 only)")
    ap.add_argument("--train", type=int, default=0, help="data-parallel training step instead of independent views")
    ap.add_argument("--views-per-step", type=int, default=2, help="--train: views per rank per optimizer step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (the render's result dict, "
                         "depth->normal map, loss, parameter gradients; --train: the updated parameters) as "
                         f"DIR/<name>.npy in float32 / float64; an array of more than {DUMP_MAX_ELEMENTS} elements as "
                         "that many of them at fixed seeded positions")
    return ap.parse_args()


DUMP_MAX_ELEMENTS = 1 << 19
DUMP_MAX_BYTES = 64 << 20
PARAM_NAMES = ("xyz", "scale", "rot", "opacity", "f_dc", "f_rest")


def collect_outputs(out, normal, loss, grads):
    """Name -> tensor of what a caller of one step receives: the render's result dict (+ the screen-space gradient),
    the depth->normal map, the loss and the gradients of the Gaussian parameters (those that have one)."""
    res = {k: v for k, v in out.items() if torch.is_tensor(v)}
    vs = out.get("viewspace_points")
    if torch.is_tensor(vs) and vs.grad is not None:
        res["viewspace_points_grad"] = vs.grad
    res["normal"], res["loss"] = normal, loss
    for name, g in zip(PARAM_NAMES, grads):
        if g is not None:
            res["grad_" + name] = g
    return res


def dump_outputs(directory, tensors):
    """Write each tensor as <directory>/<name>.npy (float64 stays float64, everything else becomes float32); a tensor of
    more than DUMP_MAX_ELEMENTS elements is written as that many of its flattened elements at sorted positions drawn
    with a fixed seed, so that two runs with the same arguments write comparable files."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    total = 0
    for name, t in tensors.items():
        t = t.detach().reshape(-1)
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise RuntimeError(f"--dump-outputs: more than {DUMP_MAX_BYTES} bytes")
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe) through NVML: a
    background thread every `period` seconds plus one sample when the host has enqueued the last step (the GPU is
    still executing the region then).  NVML is opened before the region.  (Polling `nvidia-smi -lms` from a child
    process stalled the CUDA launch path by several ms per step on these hosts; sparse NVML calls do not.)"""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, gpu_index, period=0.1):
        self.idx, self.period = gpu_index, period
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop, self._thr, self._h, self._nv = None, None, None, None

    def _phys_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip() != ""]
            if self.idx < len(ids) and ids[self.idx].strip().isdigit():
                return int(ids[self.idx])
        return self.idx

    def _sample(self):
        nv = self._nv
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for name, bit in self.REASONS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def open(self):
        """NVML initialisation (outside the timed region)."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nv = nv
            self._h = nv.nvmlDeviceGetHandleByIndex(self._phys_index())
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM))
        except Exception:
            self._h = None
        return self

    def start(self):
        import threading
        if self._h is None:
            return
        self._stop = threading.Event()

        def loop():
            while not self._stop.wait(self.period):
                self._sample()
        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def mark(self):
        """One sample now: called right after the last step was enqueued, while the GPU still executes the region."""
        if self._h is not None:
            self._sample()

    def stop(self):
        if self._h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self._stop.set()
        self._thr.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}


class HostCamera:
    """Per-view camera whose matrices live in PINNED host memory; `.upload(dev)` is the step's H2D copy."""

    def __init__(self, cam):
        self.FoVx, self.FoVy = cam.FoVx, cam.FoVy
        self.image_width, self.image_height = cam.image_width, cam.image_height
        self.h_view = cam.world_view_transform.contiguous().pin_memory()
        self.h_proj = cam.full_proj_transform.contiguous().pin_memory()
        self.h_pos = cam.camera_center.contiguous().pin_memory()
        K = cam.intrinsics
        self.fx, self.fy, self.cx, self.cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
        self.K = K
        self.nbytes = (self.h_view.numel() + self.h_proj.numel() + self.h_pos.numel()) * 4

    def upload(self, dev):
        self.world_view_transform = self.h_view.to(dev, non_blocking=True)
        self.full_proj_transform = self.h_proj.to(dev, non_blocking=True)
        self.camera_center = self.h_pos.to(dev, non_blocking=True)
        return self


class PinnedCam:
    """Camera whose matrices are still in pinned host memory (graph mode: the copy into the graph's static tensors is
    the step's H2D)."""

    def __init__(self, hc):
        self.world_view_transform, self.full_proj_transform, self.camera_center = hc.h_view, hc.h_proj, hc.h_pos


def mapped_repo_libraries():
    """In-tree shared objects this process has mapped (self-check that the reference arm runs none of ours)."""
    libs = set()
    try:
        for line in open("/proc/self/maps"):
            path = line.split()[-1]
            if path.endswith(".so") and os.path.realpath(path).startswith(os.path.realpath(ROOT) + os.sep):
                libs.add(os.path.relpath(os.path.realpath(path), os.path.realpath(ROOT)))
    except OSError:
        pass
    return sorted(libs)


def targets(dev, H, W):
    g = torch.Generator().manual_seed(1234)
    return (torch.rand(3, H, W, generator=g).to(dev), (3.0 * torch.rand(1, H, W, generator=g)).to(dev),
            torch.rand(1, H, W, generator=g).to(dev))


def make_loss(dev, H, W):
    import torch.nn.functional as F
    tc, td, to = targets(dev, H, W)

    def loss_fn(out):
        return F.l1_loss(out["render"], tc) + 0.1 * F.l1_loss(out["rendered_depth"], td) + \
            0.1 * F.l1_loss(out["rendered_final_opacity"], to)
    return loss_fn


def workload_string(cfgname, c, P, W, H, D, backward):
    scene = (f"ball rho={c.get('rho')}, s0={c.get('s0')}" if not c.get("unbounded") else
             "30% unit ball s0=0.008 + 70% shell r in [2,30]")
    what = ("fwd+bwd (L1 colour + 0.1 L1 depth + 0.1 L1 opacity) + depth->normal" if backward else
            "forward only (no_grad): colour + depth + median depth + opacity, + depth->normal")
    return (f"{cfgname}: {P} Gaussians ({scene}, seed {c['seed']}), {W}x{H}, SH degree {D}, orbit views "
            f"r={c['radius']} elev={c['elev']}, {what}")


def metric_name(cfgname, backward, custom):
    if cfgname in ("cfg3", "cfg4") and backward and not custom:
        return "views/sec fwd+bwd @1M Gaussians/1080p"
    return f"views/sec {'fwd+bwd' if backward else 'fwd-only'} ({cfgname})"


def algorithmic_bytes(P, P_vis, D, R, R_need, W, H):
    """SURVEY.md 8(d) per-view algorithmic bytes of each stage group."""
    T = ((W + 15) // 16) * ((H + 15) // 16)
    return {
        "preprocess_fwd": P * (44 + 12 * (D + 1) ** 2) + P_vis * 48,
        "binning": R * 44,
        "render_fwd": R_need * 44 + W * H * 40 + T * 8,
        "render_bwd": R_need * 44 + W * H * 40 + R_need * 40,
        "preprocess_bwd": P_vis * (300 + 304),
    }


def cpu_baseline(model, cam, D, backward):
    """CPU oracle (C++/OpenMP port of the reference algorithm) on a bounded sample of the same workload."""
    import numpy as np
    from oracle.oracle import Oracle, num_threads
    with torch.no_grad():
        x = dict(means3D=model.get_attribute("xyz").cpu().numpy(), opacities=model.get_attribute("opacity").cpu().numpy(),
                 scales=model.get_attribute("scale").cpu().numpy(), rotations=model.get_attribute("rot").cpu().numpy(),
                 shs=model.get_features.cpu().numpy(), viewmatrix=cam.h_view.numpy(), projmatrix=cam.h_proj.numpy(),
                 campos=cam.h_pos.numpy(), tanfovx=math.tan(cam.FoVx * 0.5), tanfovy=math.tan(cam.FoVy * 0.5),
                 W=cam.image_width, H=cam.image_height, sh_degree=D)
    o = Oracle()
    H, W = cam.image_height, cam.image_width
    ones = np.ones((3, H, W), np.float32)
    t0 = time.time()
    n = 0
    while True:
        o.forward(**x)
        if backward:
            o.backward(ones, ones[0], None, ones[0])
        n += 1
        if time.time() - t0 > 8.0 or n >= 4:
            break
    dt = time.time() - t0
    return {"value": n / dt, "unit": "views/s", "cores": num_threads(), "kind": "port",
            "sample": f"{n} view(s) of the same workload, {'fwd+bwd' if backward else 'forward'}, CPU oracle "
                      "(oracle/gsr_oracle.cpp, OpenMP)"}


def build_workload(a, rank, world):
    from gaustudio_b200.camera import orbit_cameras
    from gaustudio_b200.synthetic import CONFIGS, build_config
    cfgname = a.config
    scene_cfg = "cfg3" if cfgname == "cfg4" else cfgname
    # cfg4 = cfg3's scene with 800 views; a multi-GPU cfg3 run shards the same 800 orbit views
    nviews_total = CONFIGS["cfg4"]["K"] if cfgname == "cfg4" or (cfgname == "cfg3" and world > 1) else CONFIGS[cfgname]["K"]
    model, _, c = build_config(scene_cfg, P=a.gaussians, K=1)
    if a.sh_degree is not None:
        model.active_sh_degree = int(a.sh_degree)
    nv = a.steps * (a.views_per_step if a.train else 1) + a.warmup
    my_views = [(rank + world * i) % nviews_total for i in range(nv)]
    cams = orbit_cameras(nviews_total, c["radius"], c["elev"], c["W"], c["H"], c["fovx"], c["fovy"], indices=my_views)
    return model, [HostCamera(cm) for cm in cams], c, nviews_total


# =====================================================================================================================
# reference arm: the unmodified reference extension, its own op sequence, nothing of this framework's native code
# =====================================================================================================================
def run_reference(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:  # the reference has no multi-GPU path: rank 0 alone runs it, the other ranks exit without work
        return 0
    from oracle import ref_driver, ref_torch_ops
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    backward = a.config != "cfg5"
    model, hcams, c, nviews_total = build_workload(a, 0, 1)
    model.to(dev).requires_grad_(backward)
    D, H, W, P = model.active_sh_degree, c["H"], c["W"], c["P"]
    K, Wn = a.steps, a.warmup
    loss_fn = make_loss(dev, H, W)
    params = model.parameters_list()
    bg = torch.zeros(3, device=dev)  # the reference dereferences bg on the device in backward (backward.cu:586)
    last = {}

    def render(cam):
        xyz, shs, opacity, scales, rotations = ref_torch_ops.gaussian_properties(model)
        m2d = torch.zeros_like(xyz, requires_grad=backward) + 0
        rs = ref_driver.RefSettings(cam.image_height, cam.image_width, math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5),
                                    bg, 1.0, cam.world_view_transform, cam.full_proj_transform, D, cam.camera_center,
                                    False, False)
        color, radii, depth, median, opac = ref_driver.rasterize(rs, xyz, m2d, opacity, shs=shs, scales=scales,
                                                                 rotations=rotations)
        return {"render": color, "rendered_depth": depth, "rendered_final_opacity": opac, "radii": radii,
                "viewspace_points": m2d}

    def step(cam):
        if not backward:
            with torch.no_grad():
                out = render(cam)
                n = ref_torch_ops.depth2normal(out["rendered_depth"][0], cam.K)
            if a.dump_outputs:
                last.update(out=out, normal=n)
            return out["rendered_depth"].mean() + 0.0 * n[0, 0, 0]
        for p in params:
            p.grad = None
        out = render(cam)
        loss = loss_fn(out)
        loss.backward()
        n = ref_torch_ops.depth2normal(out["rendered_depth"].detach()[0], cam.K)
        if a.dump_outputs:
            last.update(out=out, normal=n)
        return loss.detach() + 0.0 * n[0, 0, 0]

    for i in range(max(Wn, 3)):
        step(hcams[i % len(hcams)].upload(dev))
    torch.cuda.synchronize(dev)
    for hc in hcams:
        hc.upload(dev)
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(dev.index).open()
    losses = torch.zeros(K, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    e0.record()
    t0 = time.perf_counter()
    for i in range(K):
        losses[i] = step(hcams[Wn + i])
    host_enqueue_ms = (time.perf_counter() - t0) * 1e3 / K
    e1.record()
    sampler.mark()
    torch.cuda.synchronize(dev)
    ms_dev = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, collect_outputs(last["out"], last["normal"], losses[K - 1], [p.grad for p in params]))

    host_loss = torch.zeros(K).pin_memory()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e2.record()
    vals = []
    for i in range(K):
        host_loss[i:i + 1].copy_(step(hcams[Wn + i].upload(dev)).reshape(1), non_blocking=True)
        if i >= 1:
            vals.append(float(host_loss[i - 1]))  # the copy is stream-ordered behind the next step's enqueue
    e3.record()
    torch.cuda.synchronize(dev)
    vals.append(float(host_loss[K - 1]))
    assert all(math.isfinite(v) for v in vals)
    ms_e2e = e2.elapsed_time(e3)
    v = K / (ms_dev * 1e-3)
    out = {
        "metric": metric_name(a.config, backward, a.gaussians is not None or a.sh_degree is not None),
        "value": v, "unit": "views/s", "n_gpus": 1, "steps": K, "warmup": Wn, "ms_per_step": ms_dev / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "impl": "reference",
        "config": {"workload": workload_string(a.config, c, P, W, H, D, backward), "views_total": nviews_total,
                   "parallelism": "single GPU (the reference has no multi-GPU path)", "streams_per_gpu": 1,
                   "launch": "eager kernel launches on the legacy default stream",
                   "l2": "inputs larger than L2 (236 MB of Gaussian parameters + 66 MB of per-view outputs vs 126 MB)",
                   "activations": "torch ops per view (reference op sequence)",
                   "forward_mode": "exact (one blocking 8-byte D2H per view, rasterizer_impl.cu:284)"},
        "clocks": clocks, "host_enqueue_ms_per_step": round(host_enqueue_ms, 4),
        "e2e": {"value": K / (ms_e2e * 1e-3), "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "ms_per_step": ms_e2e / K},
        "gpu_launches": 0,
        "cpu_baseline": {"value": v, "unit": "views/s", "cores": 1, "kind": "reference",
                         "sample": "the reference has no CPU implementation of this path: its own CUDA extension "
                                   "(unmodified sources compiled for sm_100a) driven by one host thread"},
    }
    out["native_so_loaded"] = mapped_repo_libraries()
    assert not any("libgsr_b200" in x for x in out["native_so_loaded"]), "the reference arm must not map libgsr_b200.so"
    print(json.dumps(out), flush=True)
    return 0


# =====================================================================================================================
# this framework
# =====================================================================================================================
def run_new(a):
    from gaustudio_b200 import _C, _lib, ops, parallel, renderers
    rank, local_rank, world = parallel.init_distributed()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = torch.distributed
    backward = a.config != "cfg5"
    model, hcams, c, nviews_total = build_workload(a, rank, world)
    model.to(dev).requires_grad_(backward)
    D, H, W, P = model.active_sh_degree, c["H"], c["W"], c["P"]
    K, Wn = a.steps, a.warmup
    L = _lib.lib()
    loss_fn = make_loss(dev, H, W)
    params = model.parameters_list()
    renderer = renderers.make({"name": "vanilla_renderer", "fused_activations": bool(a.fused)})
    _C.set_pipelined(bool(a.pipelined))
    last = {}

    def normal(cam, depth):
        return ops.depth2normal(depth, cam.fx, cam.fy, cam.cx, cam.cy)

    def step(cam, rend=renderer):
        if not backward:
            with torch.no_grad():
                out = rend.render(cam, model)
                n = normal(cam, out["rendered_depth"][0])
            if a.dump_outputs:
                last.update(out=out, normal=n)
            return out["rendered_depth"].mean() + 0.0 * n[0, 0, 0]
        for p in params:
            p.grad = None
        out = rend.render(cam, model)
        loss = loss_fn(out)
        loss.backward()
        n = normal(cam, out["rendered_depth"].detach()[0])
        if a.dump_outputs:
            last.update(out=out, normal=n)
        return loss.detach() + 0.0 * n[0, 0, 0]

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    if a.train:
        return run_train(a, _C, L, parallel, model, hcams, c, nviews_total, step, renderer, loss_fn, normal, rank, world, dev,
                         sync_all)

    # independent views alternate over `nstreams` CUDA streams (the allocator caches blocks per stream, so the
    # warm-up must touch every stream or the timed region would pay cudaMalloc)
    nstreams = max(1, a.streams)
    main_stream = torch.cuda.current_stream(dev)
    streams = [torch.cuda.Stream(dev) for _ in range(nstreams)] if nstreams > 1 else [main_stream]

    # one CUDA graph per stream: render (+ loss + backward) + depth->normal of a view become a single launch
    graphed = None
    if a.graph:
        try:
            from gaustudio_b200.graphs import GraphedViewStep
            post = lambda cam, out: normal(hcams[0], out["rendered_depth"].detach()[0])  # noqa: E731
            sample = [hc.upload(dev) for hc in hcams[:: max(1, len(hcams) // 6)]]
            cap = None
            if not backward:  # forward-only: size the capacity from exact-mode counts of the sample views
                _C.set_pipelined(False)
                e = torch.Tensor([])
                worst = 0
                with torch.no_grad():
                    for hc in sample:
                        worst = max(worst, exact_count(_C, model, hc, dev, D, H, W, e))
                cap = _C._quantise(worst, 1.3)
                _C.set_pipelined(bool(a.pipelined))
            first = GraphedViewStep(renderer, model, loss_fn if backward else None, sample, capacity=cap, post_fn=post)
            graphed = [first] + [GraphedViewStep(renderer, model, loss_fn if backward else None, sample[:1],
                                                 capacity=first.capacity, post_fn=post) for _ in range(nstreams - 1)]
        except Exception as ex:  # noqa: BLE001  (capture not possible here: fall back to eager launches)
            print(f"[bench] CUDA-graph capture failed ({type(ex).__name__}: {ex}); running eagerly", file=sys.stderr)
            graphed = None
            _C.set_pipelined(bool(a.pipelined))

    def run_step(i, cam):
        if graphed is None:
            return step(cam)
        gs = graphed[i % nstreams]
        res = gs(cam)
        if backward:
            return res + 0.0 * gs.extra[0, 0, 0]
        return res["rendered_depth"].mean() + 0.0 * gs.extra[0, 0, 0]

    # ---------------- warm-up (W >= 3 per stream), including the one collective with its final shape ----------------
    for i in range(max(Wn, 3 * nstreams)):
        with torch.cuda.stream(streams[i % nstreams]):
            run_step(i, hcams[i % len(hcams)].upload(dev))
    sync_all()
    for _ in range(2):
        parallel.gather_view_losses(torch.zeros(K, device=dev), K * world, rank, world)
    sync_all()

    # ---------------- leg 1: device-resident inputs ("value") ----------------
    for hc in hcams:
        hc.upload(dev)  # cameras resident in HBM before the timed region
    sampler = ClockSampler(local_rank).open()
    losses = torch.zeros(K, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    sampler.start()
    e0.record()
    t_host0 = time.perf_counter()
    if nstreams > 1:
        for st in streams:
            st.wait_stream(main_stream)
    for i in range(K):
        with torch.cuda.stream(streams[i % nstreams]):
            losses[i] = run_step(i, hcams[Wn + i])
    if nstreams > 1:
        for st in streams:
            main_stream.wait_stream(st)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / K  # host time to enqueue a step (no sync inside)
    all_losses = parallel.gather_view_losses(losses, K * world, rank, world)  # the one collective
    e1.record()
    sampler.mark()
    sync_all()
    ms_dev = parallel.barrier_max_ms(e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    assert bool(torch.isfinite(all_losses).all())
    _C.check_pipeline(wait=True)
    if a.dump_outputs and rank == 0:
        grads = [p.grad for p in params]
        if graphed is not None:  # the static outputs and gradients of the graph that replayed the last step
            gs = graphed[(K - 1) % nstreams]
            last.update(out=gs.out if backward else gs.loss, normal=gs.extra)
            grads = gs.grads if backward else []
        dump_outputs(a.dump_outputs, collect_outputs(last["out"], last["normal"], losses[K - 1], grads))

    # ---------------- leg 1b: per-kernel CUDA-event times over the same K steps (library-side events around every
    # launch on the caller's stream; eager launches, one stream).  Kept out of leg 1. ----------------
    L.gsr_profile_enable(1)
    for i in range(K):
        step(hcams[Wn + i])
    sync_all()
    ms = (ctypes.c_float * 8)()
    cn = (ctypes.c_int * 8)()
    L.gsr_profile_read(ms, cn)
    L.gsr_profile_enable(0)
    stage_ms = {STAGES[i]: (ms[i] / cn[i] if cn[i] else 0.0) for i in range(8)}
    _C.check_pipeline(wait=True)

    # ---------------- leg 2: end to end through the public API with host buffers ("e2e") ----------------
    host_loss = torch.zeros(K).pin_memory()      # pinned ring: one slot per step
    done = [torch.cuda.Event() for _ in range(K)]
    read_back = []
    lag = max(1, nstreams)  # the host stays this many steps ahead of the results it reads back
    sync_all()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    if nstreams > 1:
        for st in streams:
            st.wait_stream(main_stream)
    for i in range(K):
        with torch.cuda.stream(streams[i % nstreams]):
            # H2D of this step's inputs from pinned memory (graph mode: straight into the graph's static tensors)
            hc = PinnedCam(hcams[Wn + i]) if graphed is not None else hcams[Wn + i].upload(dev)
            host_loss[i:i + 1].copy_(run_step(i, hc).reshape(1), non_blocking=True)   # D2H of the step's result ...
            done[i].record()
        if i >= lag:                                                # ... consumed `lag` steps later, like a trainer
            done[i - lag].synchronize()                             # logging its loss: the GPU never waits for the host
            read_back.append(float(host_loss[i - lag]))
    for j in range(max(0, K - lag), K):
        done[j].synchronize()
        read_back.append(float(host_loss[j]))
    if nstreams > 1:
        for st in streams:
            main_stream.wait_stream(st)
    e3.record()
    sync_all()
    assert len(read_back) == K and all(math.isfinite(v) for v in read_back)
    ms_e2e = parallel.barrier_max_ms(e2.elapsed_time(e3), dev)
    _C.check_pipeline(wait=True)
    if graphed is not None:
        worst = max(g.max_rendered() for g in graphed)
        if worst > graphed[0].capacity:
            raise RuntimeError(f"a view needed {worst} tile instances, graph capacity is {graphed[0].capacity}")

    # ---------------- leg 3 (N=1): the drop-in path exactly as gaustudio's scripts call it ----------------
    dropin = None
    legs = 3
    if a.dropin and world == 1:
        dropin = run_dropin(a, _C, model, hcams, dev, renderers, step, K, Wn)
        legs += 2

    if world > 1 and rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return 0

    # ---------------- workload statistics for the roofline (outside the timed regions) ----------------
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    _C.set_pipelined(False)
    stats = []
    e = torch.Tensor([])
    with torch.no_grad():
        for hc in hcams[Wn:Wn + min(K, 4)]:
            stats.append(view_stats(_C, model, hc, dev, D, H, W, P, e))
    R = sum(s[0] for s in stats) / len(stats)
    R_need = sum(s[1] for s in stats) / len(stats)
    P_vis = sum(s[2] for s in stats) / len(stats)
    R_binned = sum(s[3] for s in stats) / len(stats)
    ab = algorithmic_bytes(P, P_vis, D, R_binned, R_need, W, H)  # binning bytes: the instances really moved
    grp_ms = {"preprocess_fwd": stage_ms["preprocess_fwd"],
              "binning": stage_ms["tile_scan"] + stage_ms["scatter"] + stage_ms["tile_sort"],
              "render_fwd": stage_ms["render_fwd"]}
    if backward:
        grp_ms.update(render_bwd=stage_ms["render_bwd"], preprocess_bwd=stage_ms["preprocess_bwd"])
    stages_out = {}
    traffic = {}
    tf = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tf):
        traffic = json.load(open(tf))
    for k in grp_ms:
        gbs = ab[k] / (grp_ms[k] * 1e-3) / 1e9 if grp_ms[k] > 0 else 0.0
        stages_out[k] = {"ms": round(grp_ms[k], 4), "algorithmic_MB": round(ab[k] / 1e6, 2), "GBps": round(gbs, 1),
                         "frac": round(gbs / hbm_peak, 4)}
    dom = max(grp_ms, key=lambda k: grp_ms[k])
    roof = {"kernel": dom, "bound": "hbm", "achieved": stages_out[dom]["GBps"], "peak": hbm_peak, "unit": "GB/s",
            "frac": stages_out[dom]["frac"],
            "traffic": traffic.get(dom) if a.config in ("cfg3", "cfg4") else None,
            "traffic_source": "constant from the committed ncu --set full capture (profiles/ncu_traffic.json), not "
                              "measured in this run",
            "peak_source": peak_src,
            "issue_active_pct": (traffic.get("_issue_active_pct") or {}).get(dom),
            "note": "FP32/SFU-bound compositing: HBM fraction is low by construction (DESIGN.md, Roofline honesty); "
                    "issue_active_pct = smsp__issue_active of this kernel in the committed ncu capture (a constant like "
                    "`traffic`): the resource it is actually bound by"}
    stages_out["_kernels_ms"] = {k: round(v, 4) for k, v in stage_ms.items()}
    stages_out["_workload"] = {"R": R, "R_binned": R_binned, "R_need": R_need, "P_visible": P_vis,
                               "tile_instances_first_view": stats[0][4],
                               "depth2normal_ms": round(stage_ms["depth2normal"], 4)}

    per_step = KERNELS_FWD + (KERNELS_BWD if backward else 0)
    out = {
        "metric": metric_name(a.config, backward, a.gaussians is not None or a.sh_degree is not None),
        "value": world * K / (ms_dev * 1e-3),
        "unit": "views/s", "n_gpus": a.gpus, "steps": K, "warmup": Wn,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(a.config, c, P, W, H, D, backward),
                   "views_total": nviews_total, "parallelism": f"view-sharded x{world}",
                   "streams_per_gpu": nstreams,
                   "launch": ("one CUDA graph per view, fixed binning capacity "
                              f"{graphed[0].capacity}" if graphed is not None else "eager kernel launches"),
                   "l2": "inputs larger than L2 (Gaussian parameters + per-view outputs vs 126 MB)",
                   "activations": ("fused into the projection kernel (fused_activations=True)" if a.fused else
                                   "torch ops per view (reference op sequence)"),
                   "forward_mode": "pipelined (no host sync; overflow-checked)" if a.pipelined else
                                   "exact (one blocking 8-byte D2H per view, like the reference)"},
        "clocks": clocks,
        "host_enqueue_ms_per_step": round(host_enqueue_ms, 4),  # if this is >= ms_per_step the run is host-bound
        "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "views/s",
                "h2d_bytes_per_step": hcams[0].nbytes, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K,
                "note": "every step: camera H2D from pinned memory + result D2H into a pinned ring, read on the host "
                        "`streams_per_gpu` steps later (the host blocks on step k-lag while steps k-lag+1..k run)"},
        "gpu_launches": per_step * K * legs,
        "roofline": roof,
        "stages": stages_out,
    }
    if dropin is not None:
        out["dropin"] = dropin
    out["native_so_loaded"] = mapped_repo_libraries()
    if not a.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_baseline(model, hcams[Wn], D, backward)
        except Exception as ex:  # noqa: BLE001
            out["cpu_baseline"] = {"error": str(ex)}
    print(json.dumps(out), flush=True)
    if world > 1 and dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    return 0


def exact_count(_C, model, hc, dev, D, H, W, e):
    """Binned tile instances of one exact-mode forward through the binding (un-fused inputs): what a fixed binning
    capacity has to cover."""
    view_stats(_C, model, hc, dev, D, H, W, None, e)
    return _C.last_num_binned()


def view_stats(_C, model, hc, dev, D, H, W, P, e):
    """(R, R_need, P_visible, R_binned) of one view.  R = the reference's num_rendered (tile-rect areas), R_binned = the
    instances that survive the exact tile culling and are really scattered / sorted, R_need = sum over tiles of the
    largest per-pixel n_contrib (list positions the compositing kernels consume).  P=None: R only."""
    R, *_o, radii, gb, bb, ib = _C.rasterize_gaussians(
        torch.zeros(3, device=dev), model.get_attribute("xyz"), e, model.get_attribute("opacity"),
        model.get_attribute("scale"), model.get_attribute("rot"), 1.0, e, hc.world_view_transform,
        hc.full_proj_transform, math.tan(hc.FoVx * 0.5), math.tan(hc.FoVy * 0.5), H, W, model.get_features.contiguous(), D,
        hc.camera_center, False, False)
    if P is None:
        return (R, 0, 0, 0, None)
    ex = _C.debug_export(P, W, H, R, gb, bb, ib)
    nc = ex["n_contrib"]
    Hp, Wp = (H + 15) // 16 * 16, (W + 15) // 16 * 16
    pad = torch.zeros(Hp, Wp, dtype=nc.dtype, device=dev)
    pad[:H, :W] = nc
    r_need = int(pad.view(Hp // 16, 16, Wp // 16, 16).amax(dim=(1, 3)).sum())
    n = (ex["ranges"][:, 1].long() - ex["ranges"][:, 0].long())
    tiles = {"max": int(n.max()), "mean": round(float(n.float().mean()), 1),
             "over_2048": int((n > 2048).sum()), "over_6144": int((n > 6144).sum()),
             "over_12288": int((n > 12288).sum()), "over_26624": int((n > 26624).sum())}
    return (R, r_need, int((radii > 0).sum()), ex["num_binned"], tiles)


def run_dropin(a, _C, model, hcams, dev, renderers, step, K, Wn):
    """The path gaustudio's own scripts take when this package replaces the reference's: `vanilla_renderer` with its
    default options (torch activations per view), exact forward (one blocking count read per view), the current
    stream, eager launches.  Same K views; `value` with device-resident cameras, `e2e` with the camera H2D from
    pinned memory and the loss read back every step."""
    plain = renderers.make({"name": "vanilla_renderer"})
    saved = _C.pipeline_state()
    _C.set_pipelined(False)
    try:
        for i in range(3):
            step(hcams[i % len(hcams)].upload(dev), plain)
        for hc in hcams:
            hc.upload(dev)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        losses = torch.zeros(K, device=dev)
        e0.record()
        t0 = time.perf_counter()
        for i in range(K):
            losses[i] = step(hcams[Wn + i], plain)
        host_ms = (time.perf_counter() - t0) * 1e3 / K
        e1.record()
        torch.cuda.synchronize(dev)
        ms_dev = e0.elapsed_time(e1)
        host_loss = torch.zeros(K).pin_memory()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        vals = []
        for i in range(K):
            host_loss[i:i + 1].copy_(step(hcams[Wn + i].upload(dev), plain).reshape(1), non_blocking=True)
            if i >= 1:
                vals.append(float(host_loss[i - 1]))
        e3.record()
        torch.cuda.synchronize(dev)
        vals.append(float(host_loss[K - 1]))
        assert all(math.isfinite(v) for v in vals)
        ms_e2e = e2.elapsed_time(e3)
    finally:
        _C.restore_pipeline(saved)
    return {"value": K / (ms_dev * 1e-3), "unit": "views/s", "ms_per_step": ms_dev / K,
            "e2e": {"value": K / (ms_e2e * 1e-3), "unit": "views/s", "ms_per_step": ms_e2e / K},
            "host_enqueue_ms_per_step": round(host_ms, 4),  # includes the time the host is blocked on the count read
            "speculation": dict(zip(("hits", "rebinned"), _C.speculation_stats())),
            "mode": "fused_activations=False, exact forward (its blocking count read behind the enqueued forward: capacity "
                    "guessed from the previous view, re-binned if too small), 1 stream, eager launches (--fused 0 "
                    "--streams 1 --graph 0 --pipelined 0): what gaustudio/renderers/base.py:10-63 sees"}


def run_train(a, _C, L, parallel, model, hcams, c, nviews_total, step, renderer, loss_fn, normal, rank, world, dev, sync_all):
    """Data-parallel training step (SURVEY.md 8f row 3; configs/vanilla.yaml:30-46, pipelines/optimizers/base.py:19-34).

    Per optimizer step every rank renders V = --views-per-step views (global batch V x world).  The parameter
    gradients of the first ceil(V/2) views accumulate in bucket A, the rest in bucket B; A's all_reduce is issued on
    NCCL's stream as soon as its last backward is enqueued and runs while B's views render; B's all_reduce is the
    exposed one.  One fused AdamW launch then consumes A + B (1/(V*world) scaling and zero_grad of both buckets
    folded in).  Exact synchronous SGD semantics: no stale gradients."""
    from gaustudio_b200 import optimizers
    dist = torch.distributed
    V = max(1, a.views_per_step)
    K, Wn = a.steps, a.warmup
    params = model.parameters_list()
    H, W, P = c["H"], c["W"], c["P"]
    bucketA = parallel.GradBucket(params)
    gradsA = [p.grad for p in params]
    bucketB = parallel.GradBucket(params) if V > 1 else None
    gradsB = [p.grad for p in params] if V > 1 else None
    opt = optimizers.FusedAdam([{"params": [p], "lr": lr} for p, lr in zip(params, (1.6e-4, 5e-3, 1e-3, 5e-2, 2.5e-3, 1.25e-4))],
                               betas=(0.9, 0.999), eps=1e-15, weight_decay=0.0, decoupled=True)
    nA = (V + 1) // 2
    scale = 1.0 / (V * world)

    def bind(grads):
        for p, g in zip(params, grads):
            p.grad = g

    def view_eager(cam, which):
        out = renderer.render(cam, model)
        loss = loss_fn(out)
        loss.backward()   # accumulates into the bound bucket's views
        normal(cam, out["rendered_depth"].detach()[0])
        return loss.detach()

    # one CUDA graph per bucket: render + loss + backward (accumulating into that bucket's views) + depth->normal
    graphs = None
    if a.graph:
        try:
            from gaustudio_b200.graphs import GraphedViewStep
            post = lambda cam, out: normal(hcams[0], out["rendered_depth"].detach()[0])  # noqa: E731
            sample = [hc.upload(dev) for hc in hcams[:: max(1, len(hcams) // 6)]]
            bind(gradsA)
            gA = GraphedViewStep(renderer, model, loss_fn, sample, post_fn=post, accumulate=True)
            graphs = [gA]
            if V > 1:
                bind(gradsB)
                graphs.append(GraphedViewStep(renderer, model, loss_fn, sample[:1], capacity=gA.capacity, post_fn=post,
                                              accumulate=True))
            bucketA.zero()
            if V > 1:
                bucketB.zero()
        except Exception as ex:  # noqa: BLE001
            print(f"[bench] CUDA-graph capture failed ({type(ex).__name__}: {ex}); running eagerly", file=sys.stderr)
            graphs = None

    def view(cam, which):
        if graphs is None:
            return view_eager(cam, which)
        return graphs[which](PinnedCam(cam) if not hasattr(cam, "world_view_transform") else cam)

    main_stream = torch.cuda.current_stream(dev)
    sA, sB = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def train_step(cams, comm=True):
        """The two halves of the step's views are independent (same parameters): they run on two streams, each followed by
        its bucket's all_reduce; the optimizer step joins both."""
        sA.wait_stream(main_stream)
        sB.wait_stream(main_stream)
        with torch.cuda.stream(sA):
            bind(gradsA)
            tot = 0.0
            for v in range(nA):
                tot = tot + view(cams[v], 0)
            if comm:
                bucketA.all_reduce(async_op=True)
        totB = 0.0
        if V > 1:
            with torch.cuda.stream(sB):
                bind(gradsB)
                for v in range(nA, V):
                    totB = totB + view(cams[v], 1)
                if comm:
                    bucketB.all_reduce(async_op=True)
        main_stream.wait_stream(sA)
        main_stream.wait_stream(sB)
        if comm:
            bucketA.wait()
            if V > 1:
                bucketB.wait()
        bind(gradsA)
        opt.step(grad_scale=scale, zero_grad=True, extra_grads=None if V == 1 else gradsB)
        return (tot + totB) / V

    _C.set_pipelined(bool(a.pipelined))
    cams_of = lambda s: [hcams[(Wn + s * V + v) % len(hcams)] for v in range(V)]  # noqa: E731
    for hc in hcams:
        hc.upload(dev)
    for s in range(max(3, Wn // V)):
        train_step(cams_of(s))
    sync_all()
    # timed: with communication; then cross-rank parameter identity; then the same steps without communication
    # (exposed communication = the difference; the ranks drift apart in that leg, so it comes last)
    res = {}

    def timed(comm):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for s in range(K):
            train_step(cams_of(s), comm=comm and world > 1)
        e1.record()
        sync_all()
        return parallel.barrier_max_ms(e0.elapsed_time(e1), dev) / K
    res["with_comm"] = timed(True)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"param_" + n: p for n, p in zip(PARAM_NAMES, params)})
    ident = None
    if world > 1:
        chk = torch.stack([p.detach().double().sum() for p in params] + [p.detach().double().abs().sum() for p in params])
        allc = [torch.empty_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        ident = bool(all(torch.equal(allc[0], x) for x in allc))
    res["no_comm"] = timed(False)
    _C.check_pipeline(wait=True)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    out = {"metric": "training steps/sec (cfg3, data-parallel)", "value": 1e3 / res["with_comm"], "unit": "steps/s",
           "n_gpus": a.gpus, "steps": K, "warmup": Wn, "ms_per_step": res["with_comm"], "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "views_per_sec": V * world * 1e3 / res["with_comm"],
           "config": {"workload": workload_string(a.config, c, P, W, H, model.active_sh_degree, True) +
                                  f"; {V} views per rank per optimizer step, fused AdamW",
                      "global_batch_views": V * world, "parallelism": f"data-parallel x{world}",
                      "grad_bytes_per_all_reduce": int(bucketA.flat.numel() * 4)},
           "launch": "one CUDA graph per view (gradients accumulate into the all-reduce buckets inside the graph)"
                     if graphs is not None else "eager kernel launches",
           "ms_per_step_without_comm": res["no_comm"],
           "exposed_comm_ms": res["with_comm"] - res["no_comm"],
           "params_identical_across_ranks": ident}
    print(json.dumps(out), flush=True)
    if world > 1 and dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    return run_new(a)


if __name__ == "__main__":
    sys.exit(main())

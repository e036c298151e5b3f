#!/usr/bin/env python3
"""bench.py -- throughput of the differentiable 4D Gaussian rasterizer on BASELINE.json's configurations.

Headline (default, --workload cfg3 = BASELINE.json configs[2]): forward+backward Mpixels/s @1352x1014 with 2M 4D
Gaussians (SH degree 3, temporal degree 2, 48 coefficients), one view per step per GPU.  A "step" = one render + one
backward of a view of the synthetic scene of SURVEY.md section 8(d), through the reference-facing Python API
(GaussianRasterizer + autograd over the C-ABI library).

  value   inputs resident in HBM, CUDA events, K steps after W warm-ups, max over ranks
  e2e     same call with HOST buffers: per step the camera matrices and the upstream gradient image are copied
          host->device from pinned memory (the image on a copy stream, double-buffered and issued one step ahead like a
          prefetching data loader, both arms alike) and
          the loss is read back device->host (asynchronously into pinned memory, collected one step later and before
          the clock stops, so the launch queue never drains)
  N > 1   one view per rank (weak scaling), replicated Gaussians; the gradient exchange of fdgs/dist.py inside the
          step: MAX all-reduce of the radii, ONE SUM all-reduce of the union's geometry rows + statistics, all-gather
          of the 3-float SH colour factors and local reconstruction of the summed dL_dsh rows
  --impl reference   the UNMODIFIED reference CUDA rasterizer (oracle/_ref, built from /root/reference by
          oracle/build_ref.py) on the same workload, same metric; if that .so did not travel, the CPU oracle port on a
          bounded sample.  Rank 0 only.

Other workloads (the remaining BASELINE.json configs, each for both arms):
  --workload cfg1   10k Gaussians, 256x256, forward only: GPU value + the CPU oracle timed on exactly this config
  --workload cfg2   500k Gaussians, 1352x1014, FORWARD ONLY (no_grad; the reference's evaluation path, train.py:276-345)
  --workload cfg4   "lego" shape training loop (100k points, 800x800, batch 2, L1 + Adam): iterations/s
  --workload cfg5   "flame_steak" shape: 300k Gaussians, duration [0,10], 1352x1014, 8 views per step sharded over the
                    ranks (strong scaling: the batch is fixed), gradient exchange inside the step

One JSON line on stdout (rank 0).
"""
import argparse
import importlib.util
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it
for p in (os.path.join(ROOT, "4d-gaussian-splatting_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

WORKLOADS = {
    # name: tests/helpers.py configuration + how it is run.  BASELINE.json configs[2] (cfg3) is the headline.
    "cfg1": dict(cfg=dict(P=10_000, W=256, H=256, seed=1235), mode="fwd", views=1,
                 metric="fwd Mpixels/s @256x256, 10k 4D Gaussians", desc="10k 4D Gaussians, 256x256, t=0.5, single view, forward only"),
    "cfg2": dict(cfg="cfg2", mode="fwd", views=1, metric="fwd Mpixels/s @1352x1014, 500k 4D Gaussians",
                 desc="500k 4D Gaussians, 1352x1014, forward only (no_grad)"),
    "cfg3": dict(cfg="cfg3", mode="fwdbwd", views=1, metric="fwd+bwd Mpixels/s @1352x1014, 2M 4D Gaussians",
                 desc="2M 4D Gaussians, 1352x1014, fwd+bwd, SH degree 3"),
    # cfg3 with upstream gradients for the depth, alpha and flow images too (losses on them, e.g. lambda_opa_mask > 0,
    # reference train.py:120-129): the AUX instantiation of the blend backward
    "cfg3aux": dict(cfg="cfg3", mode="fwdbwd", views=1, aux=True,
                    metric="fwd+bwd Mpixels/s @1352x1014, 2M 4D Gaussians, colour+depth+alpha+flow gradients",
                    desc="cfg3 with the loss touching the colour, depth, alpha and flow images"),
    "cfg4": dict(cfg=None, mode="train", views=2, metric="train iterations/s (lego shape: 100k points, 800x800, batch 2)",
                 desc="DNeRF 'lego' shape synthetic init, 800x800, batch of 2 views, L1 + Adam (lambda_rigid = 0)"),
    "cfg5": dict(cfg="cfg5", mode="fwdbwd", views=8, metric="fwd+bwd Mpixels/s @1352x1014, 300k 4D Gaussians, 8 views/step",
                 desc="N3V 'flame_steak' shape: 300k 4D Gaussians, duration [0,10], 1352x1014, 8 views per step"),
    "mid": dict(cfg="mid", mode="fwdbwd", views=1, metric="fwd+bwd Mpixels/s", desc="100k 4D Gaussians, 640x480 (smoke)"),
    # the whole optimisation step around the headline rasterization (SURVEY.md section 8(f)): render() over a
    # GaussianModel stand-in holding RAW parameters + photometric loss + backward + Adam
    "train3": dict(cfg="cfg3", mode="trainstep", views=1, metric="train-step Mpixels/s @1352x1014, 2M 4D Gaussians",
                   desc="cfg3 scene as a GaussianModel (raw parameters): render() + (0.8 L1 + 0.2 (1-SSIM)) + backward + Adam"),
}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        # nvidia-smi numbers the physical GPUs, CUDA numbers the visible ones: select by UUID when torch exposes it
        self.gpu = str(gpu_index)
        try:
            u = str(torch.cuda.get_device_properties(gpu_index).uuid)
            self.gpu = u if u.startswith("GPU-") else "GPU-" + u
        except Exception:
            pass
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.gpu, "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 300] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "gpu": self.gpu,
                "sm_mhz_min": min(busy) if busy else None}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_pyprep():
    """gaussian_renderer/pyprep.py by file path: importing the package would load the product's CUDA libraries, which
    must not be mapped into the reference arm's process (VERDICT r1, weak #10)."""
    path = os.path.join(ROOT, "4d-gaussian-splatting_b200", "gaussian_renderer", "pyprep.py")
    spec = importlib.util.spec_from_file_location("fdgs_pyprep_standalone", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------
def view_cameras(cfg, n, first_index=0):
    """View `first_index + k`, k < n, of a configuration: view 0 is the parity view of tests/helpers.py; the others turn
    a little about the scene centre and move in time (N3V-like multi-camera rig)."""
    from fdgs import synth
    import helpers
    base_pose = cfg.get("pose")
    cams = []
    dur = cfg.get("time_duration", 1.0)
    for k in range(first_index, first_index + n):
        if k == 0:
            R = T = None
            if base_pose is not None:
                R, T = synth.pose_from_euler(*base_pose)
            cams.append(synth.make_camera(cfg["W"], cfg["H"], timestamp=cfg.get("timestamp", 0.5),
                                          negative_fov=cfg.get("negative_fov", False), R=R, T=T))
            continue
        if base_pose is None:
            ang = math.radians(1.5 * ((k + 1) // 2) * (1 if k % 2 else -1))
            c, s = math.cos(ang), math.sin(ang)
            R = torch.tensor([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])
            centre = torch.tensor([0.0, 0.0, 6.0])
            T = centre - R.t() @ centre   # rotate about the scene centre
        else:
            yaw, pitch, roll, ex, ey, ez = base_pose
            R, T = synth.pose_from_euler(yaw + 1.5 * ((k + 1) // 2) * (1 if k % 2 else -1), pitch, roll, ex, ey, ez)
        cams.append(synth.make_camera(cfg["W"], cfg["H"], timestamp=cfg.get("timestamp", 0.5) + 0.01 * dur * k,
                                      negative_fov=cfg.get("negative_fov", False), R=R, T=T))
    return cams


class Workload:
    def __init__(self, name, device, view_ids):
        from fdgs import synth
        import helpers
        w = WORKLOADS[name]
        self.name, self.spec = name, w
        cfg = helpers.CONFIGS[w["cfg"]] if isinstance(w["cfg"], str) else w["cfg"]
        self.cfg = cfg
        cfg_built, cam0, sc_cpu, st0 = helpers.build(cfg)                 # identical on every rank
        self.P, self.W, self.H = cfg["P"], cfg["W"], cfg["H"]
        self.scene_cpu = sc_cpu
        self.scene = sc_cpu.to(device)
        self.device = device
        self.view_ids = list(view_ids)
        all_cams = view_cameras(cfg, max(self.view_ids) + 1 if self.view_ids else 1)
        self.cams = [all_cams[k] for k in self.view_ids]
        self.settings = [synth.raster_settings(c, sc_cpu, scale_modifier=cfg.get("scale_modifier", 1.0), device=device)
                         for c in self.cams]
        pin = (lambda t: t.pin_memory()) if device != "cpu" else (lambda t: t)
        self.G_host = []
        for k in self.view_ids:
            g = torch.Generator().manual_seed(cfg["seed"] + 999 + k)
            self.G_host.append(pin(torch.randn(3, self.H, self.W, generator=g)))
        self.params = {k: v.clone().requires_grad_(True) for k, v in self.scene.tensors().items() if k != "flow_2d"}
        # pinned host copies of the per-step inputs (camera) for the e2e leg
        self.cam_host = [{k: pin(st[k].cpu()) for k in ("viewmatrix", "projmatrix", "campos")} for st in self.settings]


class Runner:
    """One step (all local views: render [+ backward]) through a rasterizer API (ours or the reference's)."""

    def __init__(self, wl: Workload, impl: str, world: int, views_total: int):
        self.wl, self.impl, self.world, self.views_total = wl, impl, world, views_total
        self.backward = wl.spec["mode"] == "fwdbwd"
        self.aux = bool(wl.spec.get("aux"))
        if impl == "ours":
            from gaussian_renderer import GaussianRasterizationSettings, GaussianRasterizer
            self.Settings, self.Rasterizer = GaussianRasterizationSettings, GaussianRasterizer
        else:
            import ref_api
            self.ref_api = ref_api
        self.G_dev = [g.to(wl.device) for g in wl.G_host]
        self.copy_stream = torch.cuda.Stream(device=wl.device)
        self.res_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        self.res_ready = torch.cuda.Event()
        self.pending = False
        self.last = None
        self.keep_outputs = False      # --dump-outputs: hold the last view's rasterizer outputs (self.outputs())
        self.last_out = None
        # the exchange (and the factor path that avoids V dense dL_dsh accumulations) whenever a step has > 1 view
        self.exchange = impl == "ours" and self.backward and (world > 1 or len(wl.view_ids) > 1) and \
            os.environ.get("FDGS_DENSE_ALLREDUCE") is None
        self.exchange_info = None
        self.profile_exchange = False
        self.profile_serial = False
        # e2e leg: the upstream gradient image of a view is double-buffered on the device and uploaded one step ahead
        # on the copy stream (a data loader prefetching the next ground-truth image); every step still copies its
        # inputs host->device inside the timed region
        self.g_buf = [[torch.empty_like(g, device=wl.device) for _ in range(2)] for g in wl.G_host] if self.backward else []
        self.g_ready = [[None, None] for _ in wl.G_host]
        self.g_used = [[None, None] for _ in wl.G_host]
        self.g_step = 0

    def _raster(self, settings):
        p, sc = self.wl.params, self.wl.scene
        means2D = torch.zeros_like(p["means3D"], requires_grad=self.backward)
        if self.impl == "ours":
            out = self.Rasterizer(self.Settings(**settings))(
                means3D=p["means3D"], means2D=means2D, opacities=p["opacities"], shs=p["shs"], flow_2d=sc.flow_2d,
                ts=p["ts"], scales=p["scales"], scales_t=p["scales_t"], rotations=p["rotations"],
                rotations_r=p["rotations_r"])
        else:
            out = self.ref_api.rasterize(settings, p["means3D"], means2D, p["opacities"], p["shs"], sc.flow_2d, p["ts"],
                                         p["scales"], p["scales_t"], p["rotations"], p["rotations_r"])
        return out, means2D

    def _geometry(self):
        p = self.wl.params
        return [p[k] for k in ("means3D", "ts", "scales", "scales_t", "rotations", "rotations_r", "opacities")]

    def step(self, host_inputs: bool):
        """All local views.  host_inputs: camera + gradient image come from pinned host memory, the result goes back."""
        wl = self.wl
        for v in wl.params.values():
            v.grad = None
        cur = torch.cuda.current_stream()
        step = None
        if self.exchange:
            from fdgs.dist import ViewParallelStep
            step = ViewParallelStep(wl.P, wl.device, expected_views=len(wl.view_ids))
            step.profile = self.profile_exchange
            step.profile_serial = self.profile_serial
            step.__enter__()
        result = None
        try:
            for i in range(len(wl.view_ids)):
                st = wl.settings[i]
                G = self.G_dev[i]
                if host_inputs:
                    st = dict(st)
                    for k, h in wl.cam_host[i].items():
                        st[k] = h.to(wl.device, non_blocking=True)
                    if self.backward:
                        # the upstream gradient image (stand-in for the ground-truth image of a training step): uploaded
                        # on a copy stream, this step's copy was issued during the previous step (prefetch depth 1)
                        b = self.g_step & 1
                        if self.g_ready[i][b] is None:
                            self._upload(i, b)
                        G, ready = self.g_buf[i][b], self.g_ready[i][b]
                        self.g_ready[i][b] = None
                if self.backward:
                    (color, radii, depth, alpha, flow, covs), means2D = self._raster(st)
                    if self.keep_outputs:
                        self.last_out = dict(color=color, radii=radii, depth=depth, alpha=alpha, flow=flow, covs=covs)
                    if host_inputs:
                        cur.wait_event(ready)
                    loss = (color * G).sum() / self.views_total
                    if self.aux:
                        loss = loss + ((depth * G[:depth.shape[0]]).sum() + (alpha * G[1:1 + alpha.shape[0]]).sum() +
                                       (flow * G[:flow.shape[0]]).sum()) / self.views_total
                    loss.backward()
                    if host_inputs:
                        b = self.g_step & 1
                        ev = torch.cuda.Event()
                        ev.record(cur)
                        self.g_used[i][b] = ev          # the buffer may be overwritten once this step's kernels are done
                        self._upload(i, b ^ 1)          # next step's image, overlapping the rest of this step
                    result = loss.detach() if result is None else result + loss.detach()
                    if step is not None:
                        step.add_view_stats(means2D.grad, radii)
                    self.last = (loss, radii, means2D)
                else:
                    with torch.no_grad():
                        (color, radii, depth, alpha, flow, covs), means2D = self._raster(st)
                    if self.keep_outputs:
                        self.last_out = dict(color=color, radii=radii, depth=depth, alpha=alpha, flow=flow, covs=covs)
                    result = color.mean() if result is None else result + color.mean()
                    self.last = (result, radii, means2D)
        finally:
            if step is not None:
                step.__exit__(None, None, None)
        if step is not None:
            step.finish(self._geometry(), [wl.params["shs"]], views_per_rank=len(wl.view_ids))
            self.exchange_info = step.info
        elif self.impl == "ours" and self.backward and self.world > 1:
            # FDGS_DENSE_ALLREDUCE: the plain NCCL baseline (every gradient tensor, densely)
            from fdgs.dist import allreduce_gradients, ViewBatchStats
            stats = ViewBatchStats(wl.P, wl.device)
            stats.add_view(self.last[2].grad, self.last[1])
            stats.reduce()
            allreduce_gradients([v.grad for v in wl.params.values()])
        if host_inputs:
            self.g_step += 1
            # device->host read of the step's result: an asynchronous copy into pinned memory, collected at the start of
            # the next step (and by drain() before the clock stops) -- the way a training loop logs its loss without
            # stalling the launch queue.  Every step's result is read inside the timed region.
            prev = self.drain()
            self.res_host.copy_(result.reshape(1), non_blocking=True)
            self.res_ready.record(cur)
            self.pending = True
            return prev
        return result

    def _upload(self, i, b):
        with torch.cuda.stream(self.copy_stream):
            if self.g_used[i][b] is not None:
                self.copy_stream.wait_event(self.g_used[i][b])
            self.g_buf[i][b].copy_(self.wl.G_host[i], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.g_ready[i][b] = ev

    def drain(self):
        """Wait for and return the most recent step's result (None if nothing is pending)."""
        if not self.pending:
            return None
        self.res_ready.synchronize()
        self.pending = False
        return float(self.res_host[0])

    def outputs(self):
        """What the last step handed its caller: the rasterizer outputs of the last view and the loss; with a backward
        also the gradients of the Gaussian parameters and of the screen-space means (summed over the step's views)."""
        out = dict(self.last_out, loss=self.last[0])
        # covariance rows of Gaussians the preprocess culled (radii 0) are never written, as in the reference: zero them
        # so that two runs or builds compare equal
        out["covs"] = torch.where((out["radii"] > 0)[:, None], out["covs"], 0.0)
        if self.backward:
            out.update({"grad_" + k: v.grad for k, v in self.wl.params.items()})
            out["grad_means2D"] = self.last[2].grad
        return out

    def h2d_bytes(self):
        cam = sum(h.numel() * 4 for c in self.wl.cam_host for h in c.values())
        img = sum(g.numel() * 4 for g in self.wl.G_host) if self.backward else 0
        return int(cam + img)


def timed(fn, steps, warmup, device, world, finish=None):
    for _ in range(warmup):
        fn()
    if finish is not None:
        finish()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        fn()
    if finish is not None:
        finish()      # e.g. collect the last step's host read-back before the clock stops
    e1.record()
    torch.cuda.synchronize(device)
    wall = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps, wall / steps * 1e3


DUMP_BYTES = 64 << 20


def dump_outputs(path, outputs, P):
    """--dump-outputs: one float32 DIR/<name>.npy per output.  When everything would exceed DUMP_BYTES, the per-Gaussian
    arrays (first dimension P) keep the same seeded sample of rows -- the largest power of two that fits -- whose
    indices go to DIR/gaussian_index.npy (float64), so that two builds can be compared output for output."""
    outputs = {k: v.detach() for k, v in outputs.items() if v is not None}
    per_gaussian = [k for k, v in outputs.items() if v.dim() > 0 and v.shape[0] == P]
    fixed = sum(4 * v.numel() for k, v in outputs.items() if k not in per_gaussian)
    row = sum(4 * outputs[k][0].numel() for k in per_gaussian)
    index = None
    if fixed + P * row > DUMP_BYTES:
        n = 1 << int(math.log2(max((DUMP_BYTES - fixed) // (row + 8), 1)))
        g = torch.Generator().manual_seed(0)
        index = torch.sort(torch.randperm(P, generator=g)[:n]).values
    os.makedirs(path, exist_ok=True)
    for k, v in outputs.items():
        if index is not None and k in per_gaussian:
            v = v[index.to(v.device)]
        np.save(os.path.join(path, k + ".npy"), v.float().cpu().numpy())
    if index is not None:
        np.save(os.path.join(path, "gaussian_index.npy"), index.double().numpy())


# ------------------------------------------------------------------------------------------------
def cpu_port_baseline():
    """The CPU oracle (port of the reference algorithm) on a bounded sample of the headline workload: a 1/8-scale
    replica with the same Gaussians-per-pixel density (250k Gaussians at 478x358), all stages, forward + backward,
    every host core the oracle can use (OpenMP in preprocess / forward blend)."""
    import oracle_py
    import helpers
    cfg, cam, sc, st = helpers.build("q250k")
    inp = helpers.oracle_inputs(st, sc, cfg)
    gc, gd, ga, gf = helpers.pixel_grads(cfg)
    z = lambda t: np.zeros_like(t.numpy())
    t0 = time.perf_counter()
    f = oracle_py.forward(inp)
    t1 = time.perf_counter()
    oracle_py.backward(inp, f, gc.numpy(), z(gd), z(ga), z(gf))
    t2 = time.perf_counter()
    mpix = cfg["W"] * cfg["H"] / 1e6
    return {"value": mpix / (t2 - t0), "unit": "Mpixels/s", "cores": oracle_py.num_threads(), "kind": "port",
            "sample": "NOT cfg3 itself: a 1/8-scale replica of it (250k Gaussians, 478x358, same density), all stages, "
                      "fwd %.2fs + bwd %.2fs" % (t1 - t0, t2 - t1)}


def cpu_cfg1_baseline():
    """BASELINE.json configs[0] exactly (10k Gaussians, 256x256, t = 0.5, forward only) on the host cores: the C oracle
    with one thread and with all of them, and the reference's python-preprocess branch (SURVEY.md section 8d, cfg1)."""
    import oracle_py
    import helpers
    cfg, cam, sc, st = helpers.build(WORKLOADS["cfg1"]["cfg"])
    inp = helpers.oracle_inputs(st, sc, cfg)
    mpix = cfg["W"] * cfg["H"] / 1e6
    out = {"config": "10k 4D Gaussians, 256x256, t=0.5, forward only (BASELINE.json configs[0])", "os_cpu_count": os.cpu_count()}
    for label, nthr in (("all_threads", None), ("one_thread", 1)):
        try:
            if nthr is not None:
                oracle_py.set_num_threads(nthr)
            oracle_py.forward(inp)                     # warm (page-in)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                oracle_py.forward(inp)
                ts.append(time.perf_counter() - t0)
            out[label] = {"ms": 1e3 * float(np.median(ts)), "Mpixels/s": mpix / float(np.median(ts)),
                          "threads": oracle_py.num_threads()}
        except AttributeError:
            out[label] = None
        finally:
            if nthr is not None and hasattr(oracle_py, "set_num_threads"):
                oracle_py.set_num_threads(0)
    pyprep = load_pyprep()
    xyzt = torch.cat([sc.scales, sc.scales_t], 1)
    with torch.no_grad():
        t0 = time.perf_counter()
        pyprep.python_preprocess(sc.means3D, sc.ts, xyzt, sc.rotations, sc.rotations_r, sc.opacities, sc.shs,
                                 cam.camera_center, cam.timestamp, sc.time_duration, 3, 2)
        out["python_preprocess_ms"] = 1e3 * (time.perf_counter() - t0)
    out["torch_threads"] = torch.get_num_threads()
    return out


def python_preprocess_baseline(wl: Workload, max_points=2_000_000):
    """The reference's Python preprocess branches (compute_cov3D_python + convert_SHs_python,
    gaussian_renderer/__init__.py:73-81,98-111) restated device-agnostically and timed on the host cores."""
    pyprep = load_pyprep()
    sc = wl.scene_cpu
    n = min(sc.P, max_points)
    xyzt = torch.cat([sc.scales[:n], sc.scales_t[:n]], 1)
    cam = wl.cams[0]
    t0 = time.perf_counter()
    with torch.no_grad():
        pyprep.python_preprocess(sc.means3D[:n], sc.ts[:n], xyzt, sc.rotations[:n], sc.rotations_r[:n], sc.opacities[:n],
                                 sc.shs[:n], cam.camera_center, cam.timestamp, sc.time_duration, 3, 2)
    dt = time.perf_counter() - t0
    return {"ms": dt * 1e3, "gaussians": n, "threads": torch.get_num_threads(), "cores": os.cpu_count()}


def parity_block(wl: Workload, reruns=4):
    """PSNR / bit-equality of the image and per-gradient error of OUR arm against the compiled reference on the
    workload's first view (outside every timed region); the reference's own run-to-run spread next to it."""
    import oracle_py
    import helpers
    import fdgs
    if not oracle_py.ref_available():
        return {"available": False, "why": "oracle/_ref/ref_rasterizer.so not present"}
    ref = oracle_py.ref_module()
    C = fdgs.ext()
    st, sc, cfg = wl.settings[0], wl.scene, wl.cfg
    dev = wl.device
    with torch.no_grad():
        fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
        rf = ref.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
        mse = float(((fw[1].double() - rf[1].double()) ** 2).mean())
        out = {"available": True, "image_bit_identical": bool(torch.equal(fw[1], rf[1])),
               "psnr_db": None if mse == 0 else 10 * math.log10(1.0 / mse), "psnr_note": "null = infinite (mse 0)",
               "radii_bit_identical": bool(torch.equal(fw[5], rf[5])),
               "tile_instances": {"ours": int(fw[0]), "reference": int(rf[0]),
                                  "note": "private scratch state: ours lists a Gaussian only in the tiles its alpha >= 1/255 "
                                          "footprint reaches (fdgs_set_tile_cull(0) reproduces the reference's lists exactly)"}}
        for i, key in ((2, "flow"), (3, "depth"), (4, "T"), (10, "out_means3D")):
            out[key + "_bit_identical"] = bool(torch.equal(fw[i], rf[i]))
        if wl.spec["mode"] != "fwdbwd":
            return out
        G = wl.G_host[0].to(dev)
        e = torch.empty(0, device=dev)
        z = lambda *s: torch.zeros(*s, device=dev)
        ours = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (G, e, e, e)))
        up = (G, z(1, wl.H, wl.W), z(1, wl.H, wl.W), z(2, wl.H, wl.W))
        runs = [ref.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, rf, up)) for _ in range(reruns)]
        grads = {}
        for k, name in enumerate(helpers.GRAD_NAMES):
            rs = [r[k] for r in runs]
            if rs[0].numel() == 0 or name in ("dL_dcov3D", "dL_dcolors", "dL_dflows"):
                continue
            m = torch.stack([r.double() for r in rs]).mean(0)
            nm = float(m.norm())
            if nm == 0:
                continue
            l2 = float((ours[k].double() - m).norm()) / nm
            spread = float(np.sqrt(np.mean([(float((r.double() - m).norm()) / nm) ** 2 for r in rs])))
            grads[name] = {"l2_vs_ref_mean": l2, "ref_run_spread_l2": spread}
        out["gradients"] = grads
        out["reference_reruns"] = reruns
        out["worst_l2"] = max(v["l2_vs_ref_mean"] for v in grads.values())
    return out


# ------------------------------------------------------------------------------------------------
def run_train(args, rank, device):
    """--workload cfg4: iterations/s of the lego-shape optimisation loop (tests/lego.py), ours or the reference."""
    import lego
    impl = "ours" if args.impl == "ours" else "ref"
    P, W, H, batch = 100_000, 800, 800, 2
    cams, init, teacher = lego.lego_setup(P, W, H, seed=4)
    cams = [c.to(device) for c in cams]
    with torch.no_grad():
        tm = lego.LegoModel({k: v.to(device) for k, v in teacher.items()})
        gts = [lego.lego_render(tm, c, impl).clone() for c in cams]
    raw = {k: v.clone().to(device).requires_grad_(True) for k, v in init.items()}
    model = lego.LegoModel(raw)
    opt = lego.make_optimizer(raw)
    it = [0]
    losses = []

    lam_rigid = 1.0 if args.rigid else 0.0

    def one():
        losses.append(lego.train_iteration(model, opt, cams, gts, it[0], batch, impl, device, lambda_rigid=lam_rigid))
        it[0] += 1

    sampler = ClockSampler(int(device.split(":")[1]))
    sampler.start()
    ms, wall = timed(one, args.steps, args.warmup, device, 1)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict({"param_" + k: v for k, v in raw.items()}, loss=losses[-1]), P)
    curve = [float(x) for x in torch.stack(losses).cpu()]
    return {"metric": WORKLOADS["cfg4"]["metric"], "value": 1e3 / ms, "unit": "it/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg4: " + WORKLOADS["cfg4"]["desc"], "pixels_per_iteration": batch * W * H,
                       "lambda_rigid": lam_rigid,
                       "note": ("lambda_rigid = 1.0 (configs/dnerf/lego.yaml:58): k = 20 neighbours per view; ours = uniform-grid "
                                "search, reference arm = the brute-force scan of pointops2's knnquery run through csrc/knn.cu")
                               if lam_rigid else "lambda_rigid = 0 in this run (--rigid turns the kNN rigidity loss on)"},
            "Mpixels_per_s": batch * W * H / 1e6 / (ms * 1e-3), "loss_first": curve[0], "loss_last": curve[-1],
            "clocks": clocks, "wall_ms_per_step": wall,
            "e2e": {"value": 1e3 / ms, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "training loop: ground-truth images resident, loss not read back per step"}}


def run_train_step(args, rank, device):
    """--workload train3: one full optimisation step at the headline size through the reference-facing render().
    ours     : render() takes the raw-parameter entry (activations + SH concatenation in the kernels), the fused
               L1 + SSIM loss (fdgs.loss) and the fused multi-tensor Adam (fdgs.optim, dense = torch semantics);
    reference: the same Python prologue with torch getters (exp / sigmoid / F.normalize / torch.cat), the compiled
               reference rasterizer, the reference's l1_loss + ssim formula on cuDNN convolutions, torch.optim.Adam."""
    import helpers
    import lego
    from raw_model import RawModel, Pipe
    cfg, cam, sc, st = helpers.build("cfg3", device=device)
    cam = cam.to(device)
    model = RawModel(sc, seed=1, requires_grad=True)
    g = torch.Generator().manual_seed(5)
    gt = torch.rand(3, cfg["H"], cfg["W"], generator=g).to(device)
    bg = torch.zeros(3, device=device)
    lv = model.leaves()
    lrs = dict(xyz=1.6e-4, t=1.6e-4, scaling=5e-3, scaling_t=5e-3, rotation=1e-3, rotation_r=1e-3, opacity=5e-2,
               features_dc=2.5e-3, features_rest=2.5e-3 / 20)     # arguments/__init__.py defaults
    groups = [{"params": [lv[k]], "lr": lrs[k], "name": k} for k in lv]
    lam = 0.2
    if args.impl == "ours":
        from gaussian_renderer import render
        from fdgs.loss import l1_ssim_loss
        from fdgs.optim import FusedAdam
        opt = FusedAdam(groups, eps=1e-15)

        def one():
            pkg = render(cam, model, Pipe(), bg)
            loss = l1_ssim_loss(pkg["render"], gt, lam)
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return loss
    else:
        opt = torch.optim.Adam(groups, lr=0.0, eps=1e-15)

        def one():
            pkg = lego.ref_render(cam, model, bg)
            img = pkg["render"]
            loss = (1.0 - lam) * (img - gt).abs().mean() + lam * (1.0 - lego.ssim_torch(img[None], gt[None]))
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return loss

    last = [None]

    def step():
        last[0] = one()

    sampler = ClockSampler(int(device.split(":")[1]))
    sampler.start()
    ms, wall = timed(step, args.steps, args.warmup, device, 1)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict({"param_" + k: v for k, v in lv.items()}, loss=last[0]), cfg["P"])
    mpix = cfg["W"] * cfg["H"] / 1e6
    # phase breakdown (CUDA events around the phases of a few extra steps)
    phases = {}
    if args.impl == "ours":
        from gaussian_renderer import render
        from fdgs.loss import l1_ssim_loss
        ev = lambda: torch.cuda.Event(enable_timing=True)
        acc = {"render": 0.0, "loss": 0.0, "backward": 0.0, "adam": 0.0}
        import fdgs
        fdgs.profile_enable(True)
        for _ in range(3):
            e = [ev() for _ in range(5)]
            e[0].record(); pkg = render(cam, model, Pipe(), bg)
            e[1].record(); loss = l1_ssim_loss(pkg["render"], gt, lam)
            e[2].record(); loss.backward()
            e[3].record(); opt.step(); opt.zero_grad(set_to_none=True)
            e[4].record()
            torch.cuda.synchronize(device)
            for i, k in enumerate(acc):
                acc[k] += e[i].elapsed_time(e[i + 1]) / 3
        prof = fdgs.profile_read()
        fdgs.profile_enable(False)
        acc["rasterizer_stage_ms"] = {k: (v[0] / max(v[1], 1)) for k, v in prof.items() if v[1] > 0}
        phases = acc
    return {"metric": WORKLOADS["train3"]["metric"], "value": mpix / (ms * 1e-3), "unit": "Mpixels/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "train3: " + WORKLOADS["train3"]["desc"], "lambda_dssim": lam,
                       "optimizer": "Adam eps 1e-15, 9 parameter groups (dense update)"},
            "iterations_per_s": 1e3 / ms, "loss": float(last[0]), "phase_ms": phases, "clocks": clocks, "wall_ms_per_step": wall,
            "e2e": {"value": mpix / (ms * 1e-3), "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "training step: ground-truth image resident, loss not read back per step"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--rigid", action="store_true", help="cfg4: lambda_rigid = 1.0 (kNN rigidity loss) like configs/dnerf/lego.yaml")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    spec = WORKLOADS[args.workload]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return 0                      # the reference arm runs on rank 0 alone
    ref_solo = args.impl == "reference"
    solo = ref_solo or spec["mode"] != "fwdbwd"          # forward-only and training workloads do not shard
    if solo and rank != 0:
        return 0
    if world > 1 and not solo:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
    eff_world = 1 if solo else world

    import oracle_py
    if args.impl == "reference" and not (torch.cuda.is_available() and oracle_py.ref_available()):
        # the compiled reference did not travel (or no GPU): time the CPU port on its bounded sample
        cb = cpu_port_baseline()
        line = {"impl": "reference", "metric": spec["metric"], "value": cb["value"],
                "unit": "Mpixels/s", "n_gpus": 0, "steps": 1, "warmup": 0, "ms_per_step": None, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": args.workload, "note": "oracle/_ref not available: CPU port of the reference"},
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "Mpixels/s", "h2d_bytes_per_step": 0,
                                            "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU path)"
    device = "cuda:%d" % local
    torch.cuda.set_device(device)

    if spec["mode"] in ("train", "trainstep"):
        line = run_train(args, rank, device) if spec["mode"] == "train" else run_train_step(args, rank, device)
        if args.impl == "reference":
            line["impl"] = "reference"
            line["config"]["reference"] = "unmodified reference CUDA rasterizer (oracle/_ref/ref_rasterizer.so, sm_100a)"
            line["cpu_baseline"] = {"value": None, "kind": "reference", "cores": 0, "sample": "reference arm ran its CUDA path on the GPU"}
        print(json.dumps(line))
        return 0

    # ---- views of the step: cfg3 = one per rank (weak); cfg5 = a fixed batch of 8 sharded over the ranks (strong)
    from fdgs.dist import shard_views
    if spec["views"] == 1:
        views_total = eff_world
        view_ids = [rank if not solo else 0]
        scaling = "weak"
    else:
        views_total = spec["views"]
        view_ids = shard_views(views_total, rank if not solo else 0, eff_world)
        scaling = "strong"
        assert len(view_ids) > 0, "more ranks than views"
    wl = Workload(args.workload, device, view_ids)
    runner = Runner(wl, "ours" if args.impl == "ours" else "ref", eff_world, views_total)
    runner.keep_outputs = bool(args.dump_outputs) and rank == 0
    mpix = wl.W * wl.H / 1e6

    # ---- value: resident inputs -------------------------------------------------------------------
    if args.impl == "ours":
        import fdgs
    launches0 = fdgs.launch_count() if args.impl == "ours" else 0
    sampler = ClockSampler(local)
    sampler.start()
    ms_step, wall_ms = timed(lambda: runner.step(False), args.steps, args.warmup, device, eff_world)
    clocks = sampler.stop()
    if runner.keep_outputs:
        dump_outputs(args.dump_outputs, runner.outputs(), wl.P)
        runner.keep_outputs, runner.last_out = False, None
    launches = (fdgs.launch_count() - launches0) if args.impl == "ours" else None
    value = views_total * mpix / (ms_step * 1e-3)

    # ---- e2e: host buffers ---------------------------------------------------------------------------
    ms_e2e, _ = timed(lambda: runner.step(True), args.steps, max(3, args.warmup // 2), device, eff_world, finish=runner.drain)
    e2e = {"value": views_total * mpix / (ms_e2e * 1e-3), "unit": "Mpixels/s", "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": runner.h2d_bytes(), "d2h_bytes_per_step": 4}

    # ---- scene statistics + per-stage times (separate short run, not part of the numbers above) -------
    res, radii, _ = runner.last
    P_vis = int((radii > 0).sum().item())
    stats = {"P": wl.P, "P_vis": P_vis, "N_pixels": wl.W * wl.H, "views_per_step": views_total,
             "views_this_rank": len(view_ids)}
    roofline = None
    stage_ms = None
    if args.impl == "ours":
        import helpers
        fdgs.profile_enable(True)
        for _ in range(3):
            runner.step(False)
        torch.cuda.synchronize(device)
        prof = fdgs.profile_read()
        fdgs.profile_enable(False)
        if runner.exchange:
            # phase tables of the gradient exchange (CUDA events inside ViewParallelStep.finish, 3 extra steps each):
            # phase_ms = as the step runs it (geometry all-reduce overlapped with the SH reconstruction: only its exposed
            # remainder shows); phase_serial_ms = every collective waited for where it is launched (its own duration)
            runner.profile_exchange = True
            tables = {}
            for serial in (False, True):
                runner.profile_serial = serial
                acc = {}
                for _ in range(3):
                    runner.step(False)
                    for k, v in (runner.exchange_info.get("phase_ms") or {}).items():
                        acc[k] = acc.get(k, 0.0) + v / 3
                tables[serial] = acc
            runner.profile_exchange = False
            runner.profile_serial = False
            acc = tables[True]
            runner.exchange_info = dict(runner.exchange_info, phase_ms=tables[False], phase_serial_ms=tables[True])
            n = eff_world
            ab, gb = runner.exchange_info.get("geometry_allreduce_bytes"), runner.exchange_info.get("factor_bytes_per_rank")
            if n > 1 and ab and acc.get("geometry_allreduce"):
                runner.exchange_info["geometry_allreduce_busbw_GBps"] = ab * 2 * (n - 1) / n / (acc["geometry_allreduce"] * 1e-3) / 1e9
            if n > 1 and gb and acc.get("factor_allgather"):
                runner.exchange_info["factor_allgather_busbw_GBps"] = gb * (n - 1) / (acc["factor_allgather"] * 1e-3) / 1e9
        stage_ms = {k: (v[0] / max(v[1], 1)) for k, v in prof.items() if v[1] > 0}   # per view
        C = fdgs.ext()
        with torch.no_grad():
            fw = C.rasterize_gaussians(*helpers.fwd_args(wl.settings[-1], wl.scene, wl.cfg))
            _, ranges, ncontrib = C.debug_export_binning(fw[7], fw[8], fw[0], wl.W, wl.H)
            R_ours = int(fw[0])
            # SURVEY's algorithmic bytes count the REFERENCE's (tile, Gaussian) instances (its 3-sigma tile squares);
            # the library's default lists are shorter (fdgs_set_tile_cull) -- that saving shows up as time, not as
            # a smaller numerator
            with fdgs.tile_cull(0):
                fw0 = C.rasterize_gaussians(*helpers.fwd_args(wl.settings[-1], wl.scene, wl.cfg))
                R = int(fw0[0])
                del fw0
            L = (ranges[:, 1] - ranges[:, 0]).long()
            pairs_walked = int(ncontrib.long().sum().item())
            stats.update(R=R, R_listed=R_ours, pairs_upper_bound=int(L.sum().item()) * 256, pairs_walked=pairs_walked,
                         mean_last_contributor=float(ncontrib.float().mean().item()),
                         note="R = the reference's (tile, Gaussian) instances, R_listed = the instances in our tile lists; "
                              "pairs_upper_bound = sum_tiles L_t * 256; pairs_walked = sum_pixels n_contrib (list positions a "
                              "pixel traverses up to its last contributor)")
            del fw
        N = wl.W * wl.H
        peak, peak_src = measured_peak()
        # ALGORITHMIC bytes, SURVEY.md section 8(d): B_fwd = 84 P + 655 P_vis + 72 R + 32 N; B_bwd = 52 R + 36 N + 1428 P_vis
        alg_stage = {"blend_bwd": 52.0 * R + 36.0 * N + 52.0 * P_vis, "blend_fwd": 28.0 * R + 32.0 * N,
                     "preprocess_bwd": 1376.0 * P_vis, "preprocess_fwd": 84.0 * wl.P + 655.0 * P_vis,
                     "tile_sort_pack": 32.0 * R, "bin_scatter": 12.0 * R, "bin_count_scan": 8.0 * wl.P}
        dom = max(stage_ms, key=stage_ms.get)
        alg = alg_stage.get(dom, 0.0)
        ach = alg / (stage_ms[dom] * 1e-3) / 1e9
        b_fwd = 84.0 * wl.P + 655.0 * P_vis + 72.0 * R + 32.0 * N
        b_bwd = (52.0 * R + 36.0 * N + 1428.0 * P_vis) if runner.backward else 0.0
        # bytes this implementation actually moves per view (80-byte staged records, dense dL_dsh rows): NOT the roofline basis
        moved = 84.0 * wl.P + 719.0 * P_vis + 88.0 * R_ours + 32.0 * N + ((80.0 * R_ours + 36.0 * N + 852.0 * P_vis + 576.0 * wl.P) if runner.backward else 0.0)
        traffic = None
        ncu = {}
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of that kernel, per launch, from the committed ncu capture
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            tj = ncu[dom]
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        except Exception:
            pass
        per_view_ms = ms_step / max(len(view_ids), 1)
        blend_ms = stage_ms.get("blend_fwd", 0.0) + stage_ms.get("blend_bwd", 0.0)
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "algorithmic_bytes": alg, "peak_source": peak_src,
                    "note": "dominant kernel is instruction-issue / shared-memory bound, not HBM bound (profiles/): read "
                            "pairs_per_s and issue_active next to the mandated HBM fraction",
                    "pairs_per_s": {"blend_fwd": pairs_walked / (stage_ms["blend_fwd"] * 1e-3) if stage_ms.get("blend_fwd") else None,
                                    "blend_bwd": pairs_walked / (stage_ms["blend_bwd"] * 1e-3) if stage_ms.get("blend_bwd") else None,
                                    "unit": "(pixel, Gaussian) pairs walked per second"},
                    "issue_active_pct": {k: v.get("issue_active_pct") for k, v in ncu.items() if isinstance(v, dict) and "issue_active_pct" in v},
                    "per_stage_frac": {k: alg_stage[k] / (v * 1e-3) / 1e9 / peak for k, v in stage_ms.items() if k in alg_stage and v > 0},
                    "frame": {"algorithmic_bytes": b_fwd + b_bwd, "achieved": (b_fwd + b_bwd) / (per_view_ms * 1e-3) / 1e9,
                              "frac": (b_fwd + b_bwd) / (per_view_ms * 1e-3) / 1e9 / peak,
                              "moved_bytes": moved, "basis": "SURVEY.md 8(d): B_fwd + B_bwd per view over the step time per view",
                              "blend_share_of_frame": blend_ms / max(sum(stage_ms.values()), 1e-9)}}

    # ---- parity of this arm against the reference (rank 0, N = 1), CPU baselines -------------------------------
    parity = None
    cpu_baseline = None
    py_pre = None
    if rank == 0 and eff_world == 1:
        if args.impl == "ours" and not args.no_parity:
            parity = parity_block(wl)
        if not args.no_cpu_baseline:
            if args.workload == "cfg1":
                c1 = cpu_cfg1_baseline()
                a = c1.get("all_threads") or {}
                cpu_baseline = {"value": a.get("Mpixels/s"), "unit": "Mpixels/s", "cores": a.get("threads"), "kind": "port",
                                "sample": "exactly cfg1 (10k Gaussians, 256x256, forward only), C oracle, median of 3", "cfg1": c1}
            else:
                cpu_baseline = cpu_port_baseline()
                cpu_baseline["cfg1"] = cpu_cfg1_baseline()
                py_pre = python_preprocess_baseline(wl)

    if eff_world > 1 and args.impl == "ours":
        sys.stderr.write("[bench] rank %d on %s (%s): ms/step %.3f, stage_ms %s, clocks %s\n" % (
            rank, device, os.environ.get("CUDA_VISIBLE_DEVICES", "all visible"), ms_step,
            {k: round(v, 3) for k, v in (stage_ms or {}).items()}, clocks))
    if rank == 0:
        line = {
            "metric": spec["metric"],
            "value": value, "unit": "Mpixels/s", "n_gpus": eff_world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, spec["desc"]),
                       "views_per_step": views_total, "parallelism": "dp%d over views" % eff_world,
                       "l2": "inputs exceed L2 (SH rows alone are %.2f GB)" % (wl.P * 576 / 1e9),
                       "api": "GaussianRasterizer + autograd (reference-facing Python API over the C-ABI)"
                              if runner.backward else "GaussianRasterizer under no_grad (reference-facing Python API over the C-ABI)"},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "stats": stats,
            "wall_ms_per_step": wall_ms,
        }
        if runner.exchange_info is not None:
            line["exchange"] = runner.exchange_info
        if args.impl == "reference":
            line["impl"] = "reference"
            line["config"]["reference"] = "unmodified reference CUDA rasterizer (oracle/_ref/ref_rasterizer.so, sm_100a)"
            line["gpu_launches"] = None
            line["cpu_baseline"] = cpu_baseline or {"value": None, "kind": "reference", "cores": 0,
                                                    "sample": "reference arm ran its CUDA path on the GPU"}
        else:
            line["roofline"] = roofline
            line["stage_ms"] = stage_ms
            line["cpu_baseline"] = cpu_baseline
            line["parity"] = parity
        if py_pre is not None:
            line["python_preprocess_host"] = py_pre
        print(json.dumps(line))
    if world > 1 and not solo:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""bench.py — Mrays/s and frames/s of the raytracing_rb hot path on 1/2/4/8 B200.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                    # + a seeded sample of the last timed step's frames

HEADLINE.  A "step" is a batch of --frames-per-step frames PER GPU of the workload BASELINE.json's metric is quoted
on (configs[1]: 1920x1080, ground plane + 16 spheres, hard shadows, 1 spp, no recursion; a camera dolly).  Metric:
Mrays/s where rays = traced rays (work-stack items passing the cut at ray_tracer.rb:52) + shadow queries (lit_area
calls from local_lights, world.rb:75), SURVEY.md 8d.  For N > 1 (torchrun, one rank per GPU) the batch's frames are
the dealing unit: a 0.1 ms frame is far too small to cut into tiles, so rank r renders frames [r*B, (r+1)*B) whole
and they are gathered into rank 0's frame slots through a CUDA-IPC peer mapping over NVLink (copy engine behind the
kernel by default).  No collective on the data path; per-GPU work is fixed as N grows (weak scaling).

BESIDE THE HEADLINE, in the same JSON line:
  * `sustained`         the same steps back to back for >= 2 s (clocks and power sampled meanwhile);
  * `configs`           (N = 1) the other four BASELINE.json configs at their stated sizes: device ms per frame,
                        Mrays/s, e2e through rtrb_submit/rtrb_wait, roofline fraction or executed tests, and a
                        same-config CPU baseline on a stated window of the frame;
  * `strong_config5`    (every N) ONE frame of config 5 as BASELINE.json states it (3840x2160, 1 024 spheres, depth 8,
                        64 spp) rendered by rank 0 alone and cut into 32x32-pixel super-tiles over all N ranks
                        (north_star's image-tile partitioning; replaces render_fork's column strips,
                        camera.rb:41-68): ms per frame both ways, the speed-up, whether the gathered frame equals
                        the solo frame byte for byte, and e2e = the assembled frame delivered to ONE pinned host
                        buffer on rank 0 (render_fork's parent, camera.rb:42-52);
  * `gather_parity`     (N > 1) SHA-256 of the frames gathered into rank 0's slots during the timed steps against
                        the same frames rendered by rank 0 alone, and the same for the tile split.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# SURVEY.md 8d algorithmic FLOP constants (add/mul = 1, FMA = 2, div/sqrt = 1, transcendental = 1)
FLOP = dict(ray=7, sphere_reject=20, sphere_accept=44, plane_reject=14, plane_accept=29, hit=82 + 2,
            lambert_per_light=24, lambert_base=15, uv=34, shadow=10, cover_sphere_none=24, cover_sphere_full=56,
            cover_sphere_pen=83 + 4, cover_plane_reject=14, cover_plane_accept=37, primary=60 + 2)


def algorithmic_flops(s):
    return (s["rays"] * FLOP["ray"]
            + (s["sphere_tests"] - s["sphere_accepts"]) * FLOP["sphere_reject"] + s["sphere_accepts"] * FLOP["sphere_accept"]
            + (s["plane_tests"] - s["plane_accepts"]) * FLOP["plane_reject"] + s["plane_accepts"] * FLOP["plane_accept"]
            + s["hits"] * FLOP["hit"] + s["lit_lights"] * FLOP["lambert_per_light"] + s["local_shaded"] * FLOP["lambert_base"]
            + s["texel_fetches"] * FLOP["uv"] + s["shadow_queries"] * FLOP["shadow"]
            + (s["cover_sphere"] - s["cover_sphere_full"] - s["cover_sphere_penumbra"]) * FLOP["cover_sphere_none"]
            + s["cover_sphere_full"] * FLOP["cover_sphere_full"] + s["cover_sphere_penumbra"] * FLOP["cover_sphere_pen"]
            + (s["cover_plane"] - s["cover_plane_accepts"]) * FLOP["cover_plane_reject"]
            + s["cover_plane_accepts"] * FLOP["cover_plane_accept"] + s["samples"] * FLOP["primary"])


class ClockSampler(threading.Thread):
    """Samples SM clocks, power and throttle reasons DURING a timed region through NVML (nvidia-ml-py), every
    ~2 ms; falls back to polling nvidia-smi when NVML is unavailable."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        self.power_w = []
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _sample(self):
        if self.nv is not None:
            nv = self.nv
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            try:
                self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for name, bit in self.REASONS:
                if mask & bit:
                    self.reasons.add(name)
        else:
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.sw_power_cap,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.hw_thermal_slowdown")
            out = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                           "--format=csv,noheader,nounits"], timeout=5).decode()
            r = [x.strip() for x in out.strip().split(",")]
            self.sm.append(float(r[0]))
            self.max_mhz = float(r[1])
            try:
                self.power_w.append(float(r[2]))
            except ValueError:
                pass
            for (name, _), v in zip(self.REASONS, r[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self._halt.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self._halt.wait(0.002)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": max(self.power_w) if self.power_w else None,
                "source": "nvml" if self.nv is not None else "nvidia-smi"}


def workload(config_id, small=False, spp=0):
    from raytracing_rb_b200 import World, scenes
    kw = {}
    if small:
        kw = dict(width=480, height=270)
    wdoc, cdoc = scenes.build(config_id, **kw)
    if spp:
        cdoc = dict(cdoc, pre_sample_times=spp, max_sample_times=spp)
    return World(wdoc), cdoc, scenes.NAMES[config_id]


def config_record(name, cdoc):
    """`config` of the JSON line: the workload only, identical in both arms (what each arm does with it is in
    `run`)."""
    return {"workload": name, "width": int(cdoc["width"]), "height": int(cdoc["height"]),
            "pre_sample_times": int(cdoc["pre_sample_times"]), "max_sample_times": int(cdoc["max_sample_times"]),
            "trace_depth": int(cdoc["trace_depth"]), "monte_carlo_diffusion_times": int(cdoc["monte_carlo_diffusion_times"]),
            "rng": "philox4x32-10 counter keyed by (pixel, sample, ray path), seed 1",
            "l2": "flushed between timed steps (256 MiB write)"}


def scene_class(world):
    """rtrb_api.cu's scene classes (FrameParams::scene_class): "one_light" = exactly one light and soft_shadow_exponent
    == 2; "lean" = that, the light's radius exactly 0 and no textured object; else "generic"."""
    if not (len(world.lights) == 1 and float(world.soft_shadow_exponent) == 2.0):
        return "generic"
    textured = any(o.texture is not None and type(o).__name__ != "Box" for o in world.world_objects)
    return "lean" if float(world.lights[0].radius) == 0.0 and not textured else "one_light"


def kernel_name(cd, n_spheres, klass="generic"):
    """The kernel build and template instantiation rtrb_launch_trace_pre_fast dispatches this frame to
    (rtrb_trace_fast.cu): namespace = scene / frame class, template arguments = <stack capacity, DETAIL, BVH>."""
    bvh = "true" if n_spheres > 32 else "false"
    if cd.trace_depth <= 1:
        return "%s::trace_pre_fast_kernel<1,false,%s>" % ("rtrb_fast_lean" if klass == "lean" else "rtrb_fast", bvh)
    need = cd.trace_depth * (1 + cd.monte_carlo_diffusion_times) + 1
    cap = 10 if need <= 10 else 32 if need <= 32 else 128
    ns = "rtrb_fast"
    if klass in ("one_light", "lean") and cap <= 32:
        ns = "rtrb_fast_l1n" if cd.monte_carlo_diffusion_times == 0 else "rtrb_fast_l1"
    return "%s::trace_pre_tree_kernel<%d,false,%s>" % (ns, cap, bvh)


# ---- CPU legs: the reference algorithm on the host cores ----------------------------------------------------------
def cpu_window(W, H, fraction, cores):
    ww = min(W, max(1, int(round(W * fraction))))
    x0 = (W - ww) // 2
    return (x0, 0, x0 + ww, H)


def cpu_sample(world, cd, fraction, seconds, max_passes=50):
    """The FP64 C++ restatement (oracle/, `kind: port`: no Ruby interpreter exists in this image) over a centred
    full-height column strip of the frame, split into column strips over every host core exactly like render_fork
    (camera.rb:53-65).  Returns (Mrays/s, cores, passes, window, seconds)."""
    from raytracing_rb_b200 import make_opts
    from oracle import oracle
    cores = os.cpu_count() or 1
    sc = oracle.OracleScene(world.to_scene_desc())
    win = cpu_window(cd.width, cd.height, fraction, cores)
    o = make_opts(seed=1, window=win)
    t0 = time.perf_counter()
    n, rays = 0, 0
    while True:
        f = sc.render(cd, o, threads=cores, want_rgb=False, want_hit=False)
        rays += f.stats["rays"] + f.stats["shadow_queries"]
        n += 1
        if time.perf_counter() - t0 > seconds or n >= max_passes:
            break
    dt = time.perf_counter() - t0
    return rays / dt / 1e6, cores, n, win, dt


def cpu_baseline_record(world, cd, fraction, seconds):
    v, cores, n, win, dt = cpu_sample(world, cd, fraction, seconds)
    return {"value": v, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": "%d pass(es) in %.1f s over the window x in [%d,%d) of %dx%d (%.2f %% of the frame's columns, full height), "
                      "%d column strips (render_fork shape)" % (n, dt, win[0], win[2], cd.width, cd.height,
                                                               100.0 * (win[2] - win[0]) / cd.width, cores)}


def run_reference(args, rank, world_size):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores.  No Ruby
    interpreter exists in this image (probed below), so it is the FP64 C++ restatement (oracle/, `kind: port`), run
    as column strips over every host core like render_fork.  One step renders ONE frame of the workload (or the
    stated window of it); the metric is a rate, so it compares with the GPU arm's batches."""
    if rank != 0:
        return
    from raytracing_rb_b200 import Camera, make_opts
    from oracle import oracle
    world, cdoc, name = workload(args.config, args.small, args.spp)
    cd = Camera(world, cdoc).camera_desc()
    cores = os.cpu_count() or 1
    sc = oracle.OracleScene(world.to_scene_desc())
    W, H = cd.width, cd.height
    win = cpu_window(W, H, args.cpu_fraction, cores)
    opts = make_opts(seed=1, window=win)
    for _ in range(args.warmup):
        sc.render(cd, opts, threads=cores, want_rgb=False, want_hit=False)
    t0 = time.perf_counter()
    rays = 0
    for _ in range(args.steps):
        f = sc.render(cd, opts, threads=cores, want_rgb=False, want_hit=False)
        rays += f.stats["rays"] + f.stats["shadow_queries"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:  # the window the step rendered
        dump_frames(args.dump_outputs, f.rgba[None, :, win[0]:win[2]], x0=win[0])
    value = rays / dt / 1e6
    frac = (win[2] - win[0]) / W
    sample = "window x in [%d,%d) of %dx%d (%.0f%% of the frame) per step, %d column strips" % (
        win[0], win[2], W, H, 100.0 * frac, cores)
    ruby = subprocess.call("command -v ruby", shell=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) == 0
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_record(name, cdoc),
        "run": {"frames_rendered_per_step": frac, "host": "CPU only, rank 0 only", "ruby_present": ruby,
                "note": "one step = %s; Mrays/s is a rate, so it compares with the GPU arm's batched steps" % sample},
        "frames_per_s": args.steps / dt / frac if frac > 0 else None,
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def batch_cameras(world, cdoc, n, first=0):
    """Frames [first, first+n) of the fly-by: the workload's camera dollying sideways, 0.02 per frame
    (wrapping every 64 frames so every rank's share of a large batch shows the same scene content)."""
    from raytracing_rb_b200 import Camera
    cams = []
    for f in range(first, first + n):
        c = Camera(world, cdoc).camera_desc()
        c.position[1] = c.position[1] + 0.02 * (f % 64)
        cams.append(c)
    return cams


def bind_to_gpu_numa_node(index):
    """Pins this process to the CPU cores NVML reports as local to GPU `index`, BEFORE any pinned host buffer
    is allocated: on a two-socket 8-GPU box a rank whose frame buffers sit on the other socket sends every
    device-to-host frame across the inter-socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        return True
    except Exception:
        return False


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


DUMP_PIXELS = 1 << 21  # 2 Mi pixels: the two files take 48 MB


def dump_frames(out_dir, frames, x0=0):
    """`--dump-outputs`: the 8-bit frames [F, H, W, 3 or 4] a step delivered, as two float32 files in `out_dir`:
    frames_sample.npy [n, 3] (R, G, B values 0..255; the constant alpha of RGBA8 is left out) and
    frames_sample_index.npy [n, 3] (frame, y, x) of those pixels, x counted in the full frame (`frames` starts at
    column x0).  Both arms write the same layout, so their dumps pair pixel for pixel.  n = min(F*H*W, DUMP_PIXELS)
    pixels chosen with a fixed seed and kept in row-major order, so the same arguments sample the same pixels in
    every run and two builds compare output for output."""
    F, H, W, Ch = frames.shape
    n_px = F * H * W
    if n_px <= DUMP_PIXELS:
        idx = np.arange(n_px)
    else:
        idx = np.sort(np.random.default_rng(0).choice(n_px, size=DUMP_PIXELS, replace=False))
    values = frames.reshape(n_px, Ch)[idx, :3].astype(np.float32)
    f, y, x = np.unravel_index(idx, (F, H, W))
    where = np.stack([f, y, x + x0], axis=1).astype(np.float32)  # exact: every index < 2**24
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frames_sample.npy"), values)
    np.save(os.path.join(out_dir, "frames_sample_index.npy"), where)


class Ctx:
    """What every measurement below needs: torch, the rank layout, the launch stream and barrier."""

    def __init__(self, args, rank, local_rank, world_size):
        import torch
        self.torch, self.args, self.rank, self.local_rank, self.world_size = torch, args, rank, local_rank, world_size
        self.dist = None
        if world_size > 1:
            import torch.distributed as dist_mod
            self.dist = dist_mod
            # NCCL announces its version on STDOUT when the first communicator is built; stdout must carry
            # exactly one JSON line, so fd 1 points at stderr until the communicator exists
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                self.dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
                self.dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        self.stream = torch.cuda.Stream()  # a real (non-NULL) stream: NULL means "the renderer's own stream" in the C ABI
        torch.cuda.set_stream(self.stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
        self.token = torch.zeros(1, dtype=torch.int32, device="cuda")

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def device_join(self):
        """Stream-ordered cross-rank join: what follows on this rank's stream starts after everything queued so far
        on EVERY rank's stream (a 4-byte all-reduce: rendezvous only, no pixel passes through it)."""
        if self.dist is not None:
            self.dist.all_reduce(self.token)

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, vals):
        t = self.torch.tensor([float(v) for v in vals], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    def share_handle(self, handle_bytes_or_none):
        """rank 0's 64-byte CUDA-IPC handle to every rank."""
        torch = self.torch
        hbuf = torch.zeros(64, dtype=torch.uint8, device="cuda")
        if self.rank == 0:
            hbuf.copy_(torch.frombuffer(bytearray(handle_bytes_or_none), dtype=torch.uint8))
        self.dist.broadcast(hbuf, 0)
        return bytes(hbuf.cpu().numpy().tobytes())


def measure_config(ctx, config_id, frames, e2e_frames, cpu_fraction, cpu_seconds):
    """One BASELINE.json config at its stated size on this rank's GPU: device time per frame (CUDA events of the
    library around each frame's kernels, L2 flushed before every frame), Mrays/s, e2e through rtrb_submit/rtrb_wait
    with pinned host buffers, roofline fraction (brute-force algorithmic FLOPs from the STRICT counters; linear-filter
    scenes only) or executed exact tests (BVH scenes), and the same-config CPU baseline on a stated window."""
    from raytracing_rb_b200 import Camera, Renderer, _abi, make_opts, PREC_STRICT
    torch = ctx.torch
    world, cdoc, name = workload(config_id)
    cd = Camera(world, cdoc).camera_desc()
    r = Renderer(world.to_scene_desc(), ctx.local_rank)
    n_sph = sum(1 for o in world.world_objects if type(o).__name__ in ("Sphere", "Box"))
    skip = _abi.SKIP_RGB | _abi.SKIP_HIT
    o = make_opts(seed=1, skip_outputs=skip, pixel_format=_abi.FMT_RGB8)
    st, _ = r.render_device(cd, o)  # warm-up (also the counters: FAST64 counts rays / shadow queries exactly)
    rays = st["rays"] + st["shadow_queries"]
    ms = []
    for _ in range(frames):
        ctx.flush.zero_()
        torch.cuda.synchronize()
        st, _ = r.render_device(cd, o)
        ms.append(st["device_ms"])
    dev_ms = float(np.median(ms))
    rec = {"workload": name, "width": cd.width, "height": cd.height, "spp": cd.pre_sample_times,
           "ms_per_frame": dev_ms, "frames_timed": frames, "ray_queries_per_frame": rays,
           "value": rays / (dev_ms * 1e-3) / 1e6, "unit": "Mrays/s",
           "samples_per_s": st["samples"] / (dev_ms * 1e-3), "kernel": kernel_name(cd, n_sph, scene_class(world))}
    # e2e: the pipelined frame call with pinned host buffers
    bufs = [torch.empty((cd.height, cd.width, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
    eo = make_opts(seed=1, pixel_format=_abi.FMT_RGB8)
    r.wait(r.submit(cd, bufs[0], eo))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pending = []
    for i in range(e2e_frames):
        if len(pending) == 3:
            r.wait(pending.pop(0))
        pending.append(r.submit(cd, bufs[i % 3], eo))
    for t in pending:
        r.wait(t)
    dt = time.perf_counter() - t0
    rec["e2e"] = {"value": rays * e2e_frames / dt / 1e6, "unit": "Mrays/s", "ms_per_frame": dt / e2e_frames * 1e3,
                  "frames": e2e_frames, "d2h_bytes_per_frame": cd.width * cd.height * 3,
                  "api": "rtrb_submit/rtrb_wait, 3 frames in flight, pinned host buffers, rgb8"}
    if n_sph <= 32:
        # brute-force algorithmic work of the same frame (every ray tests every object): STRICT's detailed counters
        sd, _ = r.render_device(cd, make_opts(seed=1, skip_outputs=skip, precision=PREC_STRICT, count_detail=True))
        fl = algorithmic_flops(sd)
        rec["roofline"] = {"bound": "fp64", "algorithmic_flops_per_frame": fl, "achieved": fl / (dev_ms * 1e-3) / 1e12,
                           "unit": "TFLOP/s", "peak": ctx.peak64, "frac": fl / (dev_ms * 1e-3) / 1e12 / ctx.peak64 if ctx.peak64 else None}
    else:
        fd, _ = r.render_device(cd, make_opts(seed=1, skip_outputs=skip, count_detail=True))
        rec["executed"] = {"exact_fp64_tests_per_frame": fd["exact_tests"],
                           "exact_tests_per_ray_query": fd["exact_tests"] / max(1, rays),
                           "note": "BVH-filtered scene: brute-force FLOPs would be meaningless (SURVEY 8d); the tests that "
                                   "really ran and Mrays/s are reported instead"}
    if cpu_seconds > 0:
        rec["cpu_baseline"] = cpu_baseline_record(world, cd, cpu_fraction, cpu_seconds)
    r.close()
    return rec


def strong_config5(ctx, frames, spp=0, small=False):
    """north_star's multi-GPU design on the config it names: ONE frame of config 5 (3840x2160, 1 024 spheres, depth 8,
    64 spp) (a) by rank 0 alone and (b) cut into 32x32-pixel super-tiles dealt round-robin over all ranks, every
    rank's kernel storing its pixels straight into rank 0's framebuffer through a CUDA-IPC peer mapping (NVLink; no
    collective, no reduction).  Reports both frame times (device, max over ranks), the speed-up, byte equality of
    the two frames, and e2e = wall time until the ASSEMBLED frame is in one pinned host buffer on rank 0."""
    from raytracing_rb_b200 import Camera, Renderer, _abi, ipc_open, make_opts
    torch, rank, N = ctx.torch, ctx.rank, ctx.world_size
    world, cdoc, name = workload(5, small, spp)
    cd = Camera(world, cdoc).camera_desc()
    W, H = cd.width, cd.height
    r = Renderer(world.to_scene_desc(), ctx.local_rank)
    nbytes = W * H * 3
    if rank == 0:
        base = r.framebuffer_ptr(W, H)
    if N > 1:
        handle = ctx.share_handle(r.framebuffer_ipc_export(W, H) if rank == 0 else None)
        if rank != 0:
            base = ipc_open(ctx.local_rank, handle)
    skip = _abi.SKIP_RGB | _abi.SKIP_HIT
    s = ctx.stream.cuda_stream
    solo_o = make_opts(seed=1, skip_outputs=skip, pixel_format=_abi.FMT_RGB8, stream=s, rgba_device_out=base)
    split_o = make_opts(seed=1, skip_outputs=skip, pixel_format=_abi.FMT_RGB8, stream=s, rgba_device_out=base,
                        tile_rank=rank, tile_world=N)
    host = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory().numpy() if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n):
        out = []
        for _ in range(n):
            ctx.flush.zero_()
            ctx.barrier()
            ev0.record(ctx.stream)
            fn()
            ev1.record(ctx.stream)
            ctx.barrier()
            out.append(ctx.max_over_ranks(ev0.elapsed_time(ev1)))
        return float(np.median(out))

    # (a) rank 0 alone
    rays = 0
    if rank == 0:
        st, _ = r.render_device(cd, solo_o)  # warm-up + counters
        rays = st["rays"] + st["shadow_queries"]
    ms_solo = timed(lambda: r.render_device(cd, solo_o, want_stats=False) if rank == 0 else None, frames)
    solo_sha = None
    if rank == 0:
        r.framebuffer_copy_async(nbytes, host, s)
        torch.cuda.synchronize()
        solo_sha = sha(host)
        host[...] = 0
    # (b) tiles over all ranks (the framebuffer is cleared first so stale solo pixels cannot pass for gathered ones)
    ctx.barrier()
    if rank == 0:
        from raytracing_rb_b200._lib import lib
        clear = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        r.peer_push(clear.data_ptr(), base, nbytes, s)
        r.peer_push_join(s)
    ctx.barrier()
    r.render_device(cd, split_o, want_stats=False)  # warm-up (tile table upload)
    ctx.barrier()
    ms_split = timed(lambda: r.render_device(cd, split_o, want_stats=False), frames)
    # e2e: kernels on every rank -> stream-ordered join -> ONE device-to-host copy of the assembled frame on rank 0
    e2e = []
    for _ in range(frames):
        ctx.barrier()
        t0 = time.perf_counter()
        r.render_device(cd, split_o, want_stats=False)
        ctx.device_join()
        if rank == 0:
            r.framebuffer_copy_async(nbytes, host, s)
        torch.cuda.synchronize()
        e2e.append(ctx.max_over_ranks((time.perf_counter() - t0) * 1e3))
    ms_e2e = float(np.median(e2e))
    rec = None
    if rank == 0:
        split_sha = sha(host)
        rec = {"workload": name, "width": W, "height": H, "spp": cd.pre_sample_times, "ray_queries_per_frame": rays,
               "frames_timed": frames, "ms_frame_solo_rank0": ms_solo, "ms_frame_split": ms_split,
               "speedup": ms_solo / ms_split if ms_split > 0 else None, "n_gpus": N,
               "mrays_s_solo": rays / (ms_solo * 1e-3) / 1e6, "mrays_s_split": rays / (ms_split * 1e-3) / 1e6,
               "pixels_equal": split_sha == solo_sha, "sha256_solo": solo_sha, "sha256_split": split_sha,
               "e2e": {"ms_per_frame": ms_e2e, "value": rays / (ms_e2e * 1e-3) / 1e6, "unit": "Mrays/s",
                       "d2h_bytes_per_frame": nbytes, "speedup_vs_solo_device": ms_solo / ms_e2e if ms_e2e > 0 else None,
                       "api": "rtrb_render_device with tile_rank/tile_world on every rank (peer stores into rank 0's "
                              "framebuffer), stream-ordered join, rtrb_framebuffer_copy_async into ONE pinned host buffer on rank 0"},
               "partition": "32x32-pixel super-tiles dealt round-robin in row-major order (rtrb_tile_partition)"}
    ctx.barrier()
    r.close()
    return rec


def run_ours(args, rank, local_rank, world_size):
    import torch
    from raytracing_rb_b200 import (Camera, Renderer, _abi, deal_frames, ipc_open, make_opts, measure_fma_peak,
                                    PREC_FAST64, PREC_STRICT)
    from raytracing_rb_b200._lib import lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world_size > 1:  # (N = 1 keeps every host core: the CPU baseline leg runs in this process)
        bind_to_gpu_numa_node(local_rank)
    ctx = Ctx(args, rank, local_rank, world_size)
    dist, stream, barrier = ctx.dist, ctx.stream, ctx.barrier
    precision = PREC_STRICT if args.precision == "strict" else PREC_FAST64
    fmt = _abi.FMT_RGB8 if args.pixel_format == "rgb8" else _abi.FMT_RGBA8
    bpp = 3 if fmt == _abi.FMT_RGB8 else 4
    world, cdoc, name = workload(args.config, args.small, args.spp)
    B = max(1, args.frames_per_step)
    tile_split = bool(args.tile_split) and world_size > 1
    # frames this rank renders per step, and the slot each lands in inside rank 0's framebuffer
    if tile_split:
        cams = batch_cameras(world, cdoc, B)            # every rank: its tiles of the same B frames
        slots = list(range(B))
        n_slots = B
    else:
        dealt = deal_frames(rank, world_size, B)        # rank r: frames [r*B, (r+1)*B), whole
        cams = batch_cameras(world, cdoc, B, dealt[0][0] if dealt else 0)
        slots = [slot for _, slot in dealt]
        n_slots = B * world_size
    W, H = cams[0].width, cams[0].height
    slot_bytes = W * H * 4           # slots are sized for RGBA8 whatever the format
    frame_bytes = W * H * bpp
    r = Renderer(world.to_scene_desc(), local_rank)
    n_sph = sum(1 for o in world.world_objects if type(o).__name__ in ("Sphere", "Box"))

    # ---- where the pixels go: frame slots in rank 0's framebuffer (a peer mapping for the others) ----
    if rank == 0:
        base_ptr = r.framebuffer_ptr(W, H * n_slots)
    if world_size > 1:
        handle = ctx.share_handle(r.framebuffer_ipc_export(W, H * n_slots) if rank == 0 else None)
        if rank != 0:
            base_ptr = ipc_open(local_rank, handle)
    use_copy = (not tile_split) and world_size > 1 and rank != 0 and args.gather == "copy"
    local_ptr = r.framebuffer_ptr(W, H * B) if use_copy else None

    def opts(f, detail=False, prec=None):
        out = (local_ptr + f * slot_bytes) if use_copy else (base_ptr + slots[f] * slot_bytes)
        return make_opts(seed=1, precision=precision if prec is None else prec,
                         tile_rank=rank if tile_split else 0, tile_world=world_size if tile_split else 1,
                         count_detail=detail, stream=stream.cuda_stream, rgba_device_out=out,
                         skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT, pixel_format=fmt)

    # ---- untimed: this rank's work per batch (counters) and the FMA issue peaks ----
    # The algorithmic (brute-force) operation counts come from the STRICT kernel's detailed counters:
    # FAST64 produces the same frames with fewer executed tests, which must not shrink the numerator.
    flops_batch, rays_batch = 0, 0
    n_count = B if not args.count_one else 1
    brute = n_sph <= 32 and not args.count_fast
    for f in range(n_count):
        st, _ = r.render_device(cams[f], opts(f, True, PREC_STRICT if brute else None))
        flops_batch += algorithmic_flops(st) if brute else 0
        rays_batch += st["rays"] + st["shadow_queries"]
    if n_count != B:  # heavy frames: one frame counted, the batch is B copies of its cost
        flops_batch, rays_batch = flops_batch * B, rays_batch * B
    peak64 = measure_fma_peak(local_rank, True) if rank == 0 else 0.0
    peak32 = measure_fma_peak(local_rank, False) if rank == 0 else 0.0
    ctx.peak64 = peak64

    flush = ctx.flush
    step_opts = [opts(f) for f in range(B)]

    def step():
        for f in range(B):
            r.render_device(cams[f], step_opts[f], want_stats=False)
            if use_copy:  # copy engine carries the finished frame to rank 0 while the next one renders
                r.peer_push(local_ptr + f * slot_bytes, base_ptr + slots[f] * slot_bytes, frame_bytes, stream.cuda_stream)
        if use_copy:
            r.peer_push_join(stream.cuda_stream)  # the step ends when its last frame has landed
    W_steps = max(args.warmup, 3)
    for _ in range(W_steps):
        step()
    barrier()

    # ---- timed: EXACTLY K steps, CUDA events on the launch stream, L2 flushed between steps ----
    launches0 = lib().rtrb_launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record(stream)
        step()
        ev[k][1].record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    launches = lib().rtrb_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    step_ms = torch.tensor([a.elapsed_time(b) for a, b in ev], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(step_ms, op=dist.ReduceOp.MAX)  # a step is done when its slowest rank is
    total_ms = float(step_ms.sum().item())
    rays_total, flops_total, launches_total = ctx.sum_over_ranks([rays_batch, flops_batch, launches])
    frames_total = n_slots  # frames finished per step by the whole job
    value = rays_total * args.steps / (total_ms * 1e-3) / 1e6

    # ---- --dump-outputs (outside the timed region): the frames of the last timed step, as rank 0's slots hold them ----
    if args.dump_outputs and rank == 0:
        got = np.zeros((H * n_slots, W, 4), np.uint8)
        r.framebuffer_download(W, H * n_slots, got)
        dump_frames(args.dump_outputs, got.reshape(n_slots, slot_bytes)[:, :frame_bytes].reshape(n_slots, H, W, bpp))

    # ---- gather parity (N > 1, outside the timed region): what is in rank 0's slots after the last timed step
    # against the same frames rendered by rank 0 alone into a scratch renderer ----
    gather = None
    if world_size > 1:
        barrier()
        if rank == 0:
            got = np.zeros((H * n_slots, W, 4), np.uint8)
            r.framebuffer_download(W, H * n_slots, got)
            flat = got.reshape(n_slots, slot_bytes)
            solo = Renderer(world.to_scene_desc(), local_rank)
            all_cams = batch_cameras(world, cdoc, n_slots)
            bad = []
            h_got, h_want = hashlib.sha256(), hashlib.sha256()
            for f in range(n_slots):
                want = solo.render(all_cams[f], make_opts(seed=1, precision=precision, pixel_format=fmt),
                                   want_rgb=False, want_hit=False).rgba
                g = flat[f, :frame_bytes]
                h_got.update(g.tobytes())
                h_want.update(np.ascontiguousarray(want).tobytes())
                if not np.array_equal(g, want.reshape(-1)):
                    bad.append(f)
            solo.close()
            gather = {"mode": "tiles of every frame" if tile_split else "whole frames (%s)" % args.gather,
                      "frames_checked": n_slots, "frames_differing": bad[:8], "equal": not bad,
                      "sha256_gathered": h_got.hexdigest(), "sha256_solo": h_want.hexdigest()}
        barrier()

    # ---- sustained: the same steps back to back for >= 2 s, no flush, clocks and power sampled ----
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(np.ceil(args.sustained_seconds * 1.1 / max(1e-6, total_ms / args.steps * 1e-3))))
        sam = ClockSampler(local_rank)
        if rank == 0:
            sam.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(n_sus):
            step()
        e1.record(stream)
        barrier()
        sus_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
        sc = sam.stop() if rank == 0 else None
        if rank == 0:
            sus_value = rays_total * n_sus / (sus_ms * 1e-3) / 1e6
            sustained = {"seconds": sus_ms * 1e-3, "steps": n_sus, "value": sus_value, "unit": "Mrays/s",
                         "vs_value": sus_value / value if value else None, "sm_mhz_median": sc["sm_mhz"],
                         "power_w_max": sc["power_w_max"], "reasons": sc["reasons"],
                         "note": "steps back to back on the device, no L2 flush between them (the frame batch is 100 MB, "
                                 "so consecutive steps still overwrite most of the 126 MB L2)"}

    # ---- dominant kernel alone (trace over the pre samples): library-side CUDA events, cold L2 ----
    tr = []
    for k in range(min(args.steps, 10)):
        for f in range(B if not args.count_one else 1):
            flush.zero_()
            st, _ = r.render_device(cams[f], opts(f))
            tr.append(st["trace_ms"])
    trace_ms = float(np.mean(tr))

    # ---- e2e: the public frame call with HOST buffers (pinned), copies inside the timed region ----
    # Every rank delivers the frames it rendered to its own pinned host buffers over its own PCIe link
    # through the pipelined frame API (frame i+1 renders while frame i crosses PCIe).
    cam_bytes = C.sizeof(_abi.CameraDesc) + C.sizeof(_abi.RenderOpts)
    e2e_opts = make_opts(seed=1, precision=precision, pixel_format=fmt,
                         tile_rank=rank if tile_split else 0, tile_world=world_size if tile_split else 1)
    DEPTH = 3  # frames in flight (the library allows 4)
    bufs = [torch.empty((H, W, bpp), dtype=torch.uint8).pin_memory().numpy() for _ in range(DEPTH)]

    def e2e_run(n_steps):
        pending, i = [], 0
        for _ in range(n_steps):
            for f in range(B):
                if len(pending) == DEPTH:
                    r.wait(pending.pop(0))
                pending.append(r.submit(cams[f], bufs[i % DEPTH], e2e_opts))
                i += 1
        for t in pending:
            r.wait(t)
    e2e_run(1)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    e2e_value = rays_total * args.steps / e2e_s / 1e6

    # ---- the other BASELINE configs (N = 1) and the strong-scaling record of config 5 (every N) ----
    configs, strong = None, None
    if not args.headline_only:
        if world_size == 1:
            configs = {}
            plan = {1: (20, 200, 1.0, 2.0), 3: (10, 30, 0.25, 3.0), 4: (6, 12, 0.05, 3.0)}
            for cid, (nf, ne, frac, secs) in plan.items():
                if cid != args.config:
                    configs[str(cid)] = measure_config(ctx, cid, nf, ne, frac, secs)
            if args.config != 5:
                configs["5"] = measure_config(ctx, 5, 3, 3, 8.0 / 3840.0, 4.0)
        strong = strong_config5(ctx, 3)
        if world_size == 1 and configs is not None and "5" in configs and strong is not None:
            strong["note"] = "N = 1: the split is the solo frame (one rank owns every tile)"

    if rank == 0:
        if tile_split:
            how = "32x32 px super-tiles of every frame dealt round-robin over ranks, peer stores into rank 0's framebuffer"
        elif world_size > 1:
            how = ("whole frames dealt to ranks (rank r renders frames [r*B, (r+1)*B)), gathered into rank 0's frame slots by " +
                   ("the copy engine over NVLink (rtrb_peer_push)" if args.gather == "copy" else "direct peer stores from the trace kernel"))
        else:
            how = "single GPU"
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world_size, "steps": args.steps,
            "warmup": W_steps, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if tile_split else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_record(name, cdoc),
            "run": {"step": "a batch of %d frames per GPU (camera dolly)" % B, "frames_per_step": frames_total,
                    "frames_per_step_per_gpu": B, "precision_mode": args.precision, "pixel_format": args.pixel_format,
                    "rays_per_step": rays_total, "multi_gpu": how},
            "frames_per_s": args.steps * frames_total / (total_ms * 1e-3),
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": cam_bytes * frames_total,
                    "d2h_bytes_per_step": frame_bytes * frames_total if not tile_split else frame_bytes * B * world_size,
                    "frames_per_s": args.steps * frames_total / e2e_s,
                    "api": "rtrb_submit/rtrb_wait per rank (%d frames in flight, pinned host buffers, %s)" % (DEPTH, args.pixel_format)},
            "gpu_launches": int(launches_total),
            "clocks": clocks,
            "wall_s_timed_region": wall,
        }
        kname = kernel_name(cams[0], n_sph, scene_class(world))
        if brute:
            flops_frame = flops_batch / B
            achieved = flops_frame / (trace_ms * 1e-3) / 1e12
            line["roofline"] = {
                "bound": "fp64", "kernel": kname, "achieved": achieved, "peak": peak64, "unit": "TFLOP/s",
                "frac": achieved / peak64 if peak64 else None,
                "traffic": ncu_traffic_bytes() if args.config == 2 and not args.small else None,
                "peak_source": "measured in this job: dependent-free DFMA microbenchmark (rtrb_measure_fma_peak)",
                "peak_fp32": peak32, "algorithmic_flops_per_launch": flops_frame, "kernel_ms": trace_ms,
                "ncu": ncu_record() if args.config == 2 and not args.small else None,
                "hbm": {"algorithmic_bytes_per_launch": frame_bytes, "peak_gbs": measured_hbm_gbs(),
                        "achieved_gbs": frame_bytes / (trace_ms * 1e-3) / 1e9},
                "note": "FP-issue bound path (SURVEY.md 8d): HBM traffic is the framebuffer write only; rank 0's kernel and counters",
            }
        else:
            line["roofline"] = {"bound": "fp64", "kernel": kname, "achieved": None, "peak": peak64, "unit": "TFLOP/s",
                                "frac": None, "traffic": None, "kernel_ms": trace_ms,
                                "note": "BVH-filtered scene: executed tests and Mrays/s are the figures (SURVEY 8d)"}
        if sustained is not None:
            line["sustained"] = sustained
        if gather is not None:
            line["gather_parity_detail"] = {"frames": gather, "tiles": None if strong is None else {
                "equal": strong["pixels_equal"], "sha256_gathered": strong["sha256_split"], "sha256_solo": strong["sha256_solo"]}}
            line["gather_parity"] = bool(gather["equal"] and (strong is None or strong["pixels_equal"]))
        if configs is not None:
            line["configs"] = configs
        if strong is not None:
            line["strong_config5"] = strong
        if world_size == 1:
            line["cpu_baseline"] = cpu_baseline_record(world, cams[0], args.cpu_fraction, 10.0)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def ncu_record():
    """Figures of the trace kernel from the committed `ncu --set full` capture of this workload
    (profiles/r2_traffic.json, written from profiles/r2_ncu_config2_fast.txt): DRAM bytes per launch, issue-slot and pipe
    utilisation.  None when absent."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)
        except Exception:
            continue
    return None


def ncu_traffic_bytes():
    r = ncu_record()
    return r["dram_bytes_per_launch"] if r else None


def measured_hbm_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"]
    except Exception:
        return 6650.0  # fallback stated in B200_PROFILING.md


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--frames-per-step", type=int, default=16, help="frames rendered per timed step")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--precision", default="fast64", choices=["fast64", "strict"])
    ap.add_argument("--small", action="store_true", help="480x270 variant for quick checks (not a bench value)")
    ap.add_argument("--pixel-format", default="rgb8", choices=["rgb8", "rgba8"],
                    help="8-bit frame layout delivered (rgb8: alpha is the constant 255 and stays off the wire)")
    ap.add_argument("--gather", default="copy", choices=["store", "copy"],
                    help="N > 1: how finished frames reach rank 0's slots (peer stores from the kernel / copy engine)")
    ap.add_argument("--tile-split", action="store_true",
                    help="N > 1: cut every frame of the headline steps into super-tiles across the ranks")
    ap.add_argument("--spp", type=int, default=0, help="override pre = max sample count (heavy configs at reduced cost)")
    ap.add_argument("--count-one", action="store_true", help="count rays/FLOPs on one frame of the batch only")
    ap.add_argument("--count-fast", action="store_true", help="take the counters from the FAST64 kernel (heavy configs)")
    ap.add_argument("--cpu-fraction", type=float, default=1.0, help="fraction of the frame width the CPU legs render")
    ap.add_argument("--sustained-seconds", type=float, default=2.0, help="length of the back-to-back companion run (0 = skip)")
    ap.add_argument("--headline-only", action="store_true", help="skip the per-config and strong-scaling records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed seeded sample of the pixels of the frames the last step "
                         "delivered: DIR/frames_sample.npy (R, G, B) and DIR/frames_sample_index.npy (frame, y, x), "
                         "float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world_size)
    else:
        run_ours(args, rank, local_rank, world_size)


if __name__ == "__main__":
    main()

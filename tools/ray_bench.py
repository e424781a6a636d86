"""Measures the ray-level queries (rtrb_trace_rays, rtrb_intersect_rays, rtrb_camera_rays) on one GPU and writes
profiles/ray_queries.json (or --out).  Records the GPU's name and power limit in the same run.

  1. trace_rays on config 2's 1080p camera rays (2.07 M rays, depth 1, device buffers) beside the frame's trace kernel
     (render_device's trace_ms).  The frame runs the lean class build; the ray kernels are the generic build, so the
     frame is also timed on the same scene with the light's radius set to the smallest positive double, which puts it in
     the one-light class whose depth-1 frames run the generic build;
  2. the same for config 3 (1080p, 4 spp, depth 8: 8.3 M rays against the lockstep ray-tree frame kernel);
  3. 2^22 incoherent rays (uniform origins in the scene's bounds, uniform directions) in config 5's 1024-sphere BVH
     scene: trace_rays at depth 1 and intersect_rays;
  4. the host-buffer path (numpy in, numpy out, blocking) against the device-buffer path, wall time of one call.
Kernel times are CUDA events around --iters back-to-back calls on one stream after --warmup calls.

python tools/ray_bench.py [--out profiles/ray_queries.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 << 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ray_queries.json"))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import numpy as np
    import torch
    from raytracing_rb_b200 import PREC_FAST64, Camera, World, make_opts, scenes

    if not torch.cuda.is_available():
        raise SystemExit("ray_bench needs a CUDA device")
    res = {"gpu": gpu_info(), "precision": "FAST64", "warmup": args.warmup, "iters": args.iters}

    def event_ms(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.iters

    def frame_trace_ms(cam):
        r, cd = cam.renderer(), cam.camera_desc()
        opts = make_opts(seed=1, precision=PREC_FAST64, skip_outputs=3)
        for _ in range(args.warmup):
            r.render_device(cd, opts)
        t = [r.render_device(cd, opts)[0] for _ in range(args.iters)]
        return statistics.median(s["trace_ms"] for s in t), statistics.median(s["device_ms"] for s in t)

    def camera_case(cid, label):
        wdoc, cdoc = scenes.build(cid, width=1920, height=1080)
        cam = Camera(World(wdoc), cdoc)
        r, cd = cam.renderer(), cam.camera_desc()
        rays, keys = r.camera_rays(cd, seed=1, samples=(0, cd.pre_sample_times), device_buffers=True)
        n = rays.shape[0]
        depth, mc = cd.trace_depth, cd.monte_carlo_diffusion_times
        ray_ms = event_ms(lambda: r.trace_rays(rays, depth, mc, seed=1, keys=keys, want_stats=False))
        cam_ms = event_ms(lambda: r.camera_rays(cd, seed=1, samples=(0, cd.pre_sample_times), device_buffers=True))
        f_trace, f_dev = frame_trace_ms(cam)
        rec = {"scene": label, "rays": n, "trace_depth": depth, "mc": mc,
               "trace_rays_ms": ray_ms, "camera_rays_ms": cam_ms,
               "frame_trace_ms": f_trace, "frame_device_ms": f_dev,
               "trace_rays_over_frame_trace": ray_ms / f_trace,
               "bytes_in": n * (48 + 8), "bytes_out": n * (24 + 4),
               "l2_state": "rays and keys (%.0f MB) and outputs (%.0f MB) written by the previous call: %s" % (
                   n * 56 / 1e6, n * 28 / 1e6,
                   "more than the 126 MB L2, so not held" if n * 84 > L2_BYTES else "within the 126 MB L2")}
        return cam, rays, keys, rec

    # 1. config 2, depth 1
    cam2, rays2, keys2, rec = camera_case(2, "config2 1920x1080, 1 spp, depth 1")
    wdoc, cdoc = scenes.build(2, width=1920, height=1080)
    wdoc["lights"][0]["properties"]["radius"] = 5e-324  # not the lean class: the generic depth-1 frame build
    gen = Camera(World(wdoc), cdoc)
    rec["frame_trace_ms_generic_build"], rec["frame_device_ms_generic_build"] = frame_trace_ms(gen)
    rec["trace_rays_over_frame_trace_generic_build"] = rec["trace_rays_ms"] / rec["frame_trace_ms_generic_build"]
    res["config2_camera_rays"] = rec
    print(json.dumps(rec), flush=True)

    # 2. config 3, 4 spp, depth 8
    _, _, _, rec = camera_case(3, "config3 1920x1080, 4 spp, depth 8")
    res["config3_camera_rays"] = rec
    print(json.dumps(rec), flush=True)

    # 3. incoherent rays in config 5's BVH scene
    wdoc, cdoc = scenes.build(5)
    world5 = World(wdoc)
    r5 = world5.renderer(0)
    sd = world5.to_scene_desc().desc
    pts = np.array([sd.objects[i].point[:] for i in range(sd.n_objects)])
    lo, hi = pts.min(axis=0) - 1.0, pts.max(axis=0) + 1.0
    rs = np.random.RandomState(1)
    n = 1 << 22
    d = rs.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays5 = torch.from_numpy(np.hstack([rs.uniform(lo, hi, size=(n, 3)), d])).cuda()
    rec = {"scene": "config5 world (%d objects, BVH)" % sd.n_objects, "rays": n,
           "origins": "uniform in the objects' bounding box + 1", "directions": "uniform unit",
           "trace_rays_depth1_ms": event_ms(lambda: r5.trace_rays(rays5, 1, 0, want_stats=False)),
           "intersect_rays_ms": event_ms(lambda: r5.intersect_rays(rays5)),
           "l2_state": "rays 201 MB + outputs: more than the 126 MB L2, so not held"}
    rec["trace_rays_Mrays_per_s"] = n / rec["trace_rays_depth1_ms"] / 1e3
    rec["intersect_rays_Mrays_per_s"] = n / rec["intersect_rays_ms"] / 1e3
    res["config5_incoherent"] = rec
    print(json.dumps(rec), flush=True)

    # 4. host buffers against device buffers (config 2's camera rays, one blocking call each, wall time)
    r2 = cam2.renderer()
    host_rays, host_keys = rays2.cpu().numpy(), keys2.cpu().numpy().view(np.uint32)
    walls = {"host": [], "device": []}
    for _ in range(args.warmup):
        r2.trace_rays(host_rays, 1, 0, keys=host_keys)
        r2.trace_rays(rays2, 1, 0, keys=keys2)
    for _ in range(args.iters // 2):
        t0 = time.perf_counter(); r2.trace_rays(host_rays, 1, 0, keys=host_keys); walls["host"].append(time.perf_counter() - t0)
        t0 = time.perf_counter(); r2.trace_rays(rays2, 1, 0, keys=keys2); walls["device"].append(time.perf_counter() - t0)
    rec = {"scene": "config2 1920x1080 camera rays, depth 1", "rays": int(host_rays.shape[0]),
           "host_buffers_wall_ms": statistics.median(walls["host"]) * 1e3,
           "device_buffers_wall_ms": statistics.median(walls["device"]) * 1e3,
           "host_buffers_note": "pageable numpy arrays: 116 MB to the device, 58 MB back; both calls return stats "
                                "and so synchronise"}
    rec["host_over_device"] = rec["host_buffers_wall_ms"] / rec["device_buffers_wall_ms"]
    res["host_vs_device_buffers"] = rec
    print(json.dumps(rec), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

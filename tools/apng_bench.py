"""Measures animated PNG frames (rtrb_apng_add / rtrb_submit_apng, Camera.render_animation) on one GPU at 1080p and
writes profiles/apng.json (or --out).  Records the GPU's name and power limit in the same run.

Two animations of config 2, --frames frames each: one sphere moving a little every frame ("sphere"), and the camera
orbiting the point it looks at ("orbit").  For each:
  - encoder device time per frame: the APNG kernels of rtrb_apng_add (torch.profiler, summed by kernel, mean over the
    frames and --reps animations) against the kernels of rtrb_encode_png of the same full frames; the frames are
    rendered beforehand into device memory (90 x 6.2 MB: larger than L2, so every frame is read from HBM);
  - bytes per frame against rtrb_encode_png's full frame, and the APNG file against the sum of per-frame PNG files;
  - frames/s of submit_apng against submit_png, 3 frames in flight, the animation's edit (scene update or camera move)
    before every frame in both arms, alternated twice.

python tools/apng_bench.py [--out profiles/apng.json]"""
import argparse
import json
import math
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def kernel_us(prof):
    """Summed device time (us) of the encoder's kernels, by kernel (template flag kept: <true> is the crop)."""
    out = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        m = re.search(r"(a?png_[a-z]+_kernel)(<(true|false)>)?", e.name)
        if m:
            key = m.group(1) + ("<%s>" % m.group(3) if m.group(3) else "")
            out[key] = out.get(key, 0.0) + e.device_time
    return out


def rotate(v, axis, a):
    """v rotated by angle a about the unit vector `axis` (Rodrigues)."""
    c, s = math.cos(a), math.sin(a)
    d = sum(x * y for x, y in zip(v, axis))
    cr = (axis[1] * v[2] - axis[2] * v[1], axis[2] * v[0] - axis[0] * v[2], axis[0] * v[1] - axis[1] * v[0])
    return tuple(v[i] * c + cr[i] * s + axis[i] * d * (1 - c) for i in range(3))


def make_animation(kind):
    """-> (camera, step) at 1080p; step(i) edits the world or the camera before frame i."""
    from raytracing_rb_b200 import Camera, Sphere, World, scenes
    from raytracing_rb_b200.vec3 import Vec3
    wdoc, cdoc = scenes.build(2, width=1920, height=1080)
    world = World(wdoc)
    cam = Camera(world, cdoc)
    if kind == "sphere":
        k = [i for i, o in enumerate(world.world_objects) if isinstance(o, Sphere)][0]
        x, y, z = world.world_objects[k].center.to_a()

        def step(i):
            world.world_objects[k].center = Vec3(x + 0.01 * (i % 40), y - 0.008 * (i % 40), z)
        return cam, step
    pos, front, up = cam.position.to_a(), cam.front.to_a(), cam.up.to_a()
    n = math.sqrt(sum(u * u for u in up))
    axis = tuple(u / n for u in up)
    target = tuple(p + 10 * f for p, f in zip(pos, front))
    rel = tuple(p - t for p, t in zip(pos, target))

    def step(i):
        a = 0.004 * (i % 40)
        cam.position = Vec3(*[t + r for t, r in zip(target, rotate(rel, axis, a))])
        cam.front = Vec3(*rotate(front, axis, a))
    return cam, step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "apng.json"))
    ap.add_argument("--frames", type=int, default=90)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pipelined", type=int, default=400)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from raytracing_rb_b200 import Apng, _abi, apng_frame_max_bytes, make_opts, png_max_bytes

    if not torch.cuda.is_available():
        raise SystemExit("apng_bench needs a CUDA device")
    res = {"gpu": gpu_info(), "size": [1920, 1080], "frames": args.frames, "animations": {}}
    RGB8 = _abi.FMT_RGB8
    for kind in ("sphere", "orbit"):
        cam, step = make_animation(kind)
        r = cam.renderer()
        W, H = cam.width, cam.height
        frames = []
        for i in range(args.frames):
            step(i)
            r = cam.renderer()
            rgb = r.render(cam.camera_desc(), make_opts(seed=1, pixel_format=RGB8), want_rgb=False, want_hit=False).rgba
            frames.append(torch.from_numpy(rgb).cuda())
        torch.cuda.synchronize()
        pngs = [r.encode_png(W, H, RGB8, src=t.data_ptr()) for t in frames]
        anim = r.apng(W, H)
        chunks = [anim.add(src=t.data_ptr()) for t in frames]
        anim.close()
        apng_bytes = len(anim.header()) + sum(len(c) for c in chunks) + len(Apng.TRAILER)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                a = r.apng(W, H)
                for t in frames:
                    a.add(src=t.data_ptr())
                a.close()
            torch.cuda.synchronize()
        apng_k = {k: v / (args.reps * args.frames) for k, v in kernel_us(prof).items()}
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                for t in frames:
                    r.encode_png(W, H, RGB8, src=t.data_ptr())
            torch.cuda.synchronize()
        png_k = {k: v / (args.reps * args.frames) for k, v in kernel_us(prof).items()}
        rec = {
            "apng_encode_device_us_per_frame": sum(apng_k.values()), "apng_kernels_us": apng_k,
            "encode_png_device_us_per_frame": sum(png_k.values()), "encode_png_kernels_us": png_k,
            "apng_frame_bytes_mean": statistics.mean(len(c) for c in chunks[1:]),
            "apng_frame0_bytes": len(chunks[0]),
            "encode_png_bytes_mean": statistics.mean(len(p) for p in pngs),
            "apng_file_bytes": apng_bytes, "sum_png_file_bytes": sum(len(p) for p in pngs),
            "l2_state": "frames in device memory, %d x %d bytes (exceeds L2)" % (args.frames, W * H * 3),
        }

        # pipelined: the same edits before every frame in both arms
        cam, step = make_animation(kind)
        r = cam.renderer()
        eo = make_opts(seed=1, pixel_format=RGB8)
        png_bufs = [torch.empty(png_max_bytes(W, H), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
        apng_bufs = [torch.empty(apng_frame_max_bytes(W, H), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]

        def run(submit, wait, bufs):
            t0, pending = time.perf_counter(), []
            for i in range(args.pipelined):
                if len(pending) == 3:
                    wait(pending.pop(0))
                step(i)
                cam.renderer()
                pending.append(submit(cam.camera_desc(), bufs[i % 3]))
            for t in pending:
                wait(t)
            return args.pipelined / (time.perf_counter() - t0)

        fps = {"submit_png": [], "submit_apng": []}
        for _ in range(2):
            fps["submit_png"].append(run(lambda cd, b: r.submit_png(cd, b, eo), r.wait_png, png_bufs))
            a = r.apng(W, H)
            fps["submit_apng"].append(run(lambda cd, b: a.submit(cd, b, eo), a.wait, apng_bufs))
            a.close()
        rec["pipelined_frames_per_s"] = {k: max(v) for k, v in fps.items()}
        rec["pipelined_frames_per_s"].update(all_runs=fps, frames=args.pipelined, in_flight=3)
        res["animations"][kind] = rec
        print(json.dumps({"animation": kind, **rec}), flush=True)
        del frames

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
